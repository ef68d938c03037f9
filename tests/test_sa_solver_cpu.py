"""CPU tests of the SA-Solver sampler: the oracle restatement (oracle/sa_oracle.py) against fixtures produced by the unmodified
reference `SASolverSampler` (oracle/gen_golden_sa.py), the product's host-side plan against the oracle's scalars, the public
surface, and the C-ABI struct of the step kernel."""
import ctypes
import inspect
import os
import subprocess
import sys
import tempfile
import types

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import sa_oracle as so              # noqa: E402
from oracle.gen_golden_sa import CASES          # noqa: E402
from pixart_sigma_b200 import lib, sampler      # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
PLAN_KEYS = ("t_input", "sigma", "inv_alpha", "cA", "c0", "c1", "cN", "pA", "p0", "p1", "pN")


def _rel(a, b):
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_matches_reference_fixture(name):
    """Same float32 operations in the same order as the reference: 1e-6 only leaves room for differences between torch builds."""
    case, g = CASES[name], torch.load(os.path.join(GOLD, name + ".pt"))
    assert len(g["noises"]) == case["steps"] + 1                        # S + 1 draws, the first one unused
    out, info = so.sample(so.toy_model, g["x_T"], g["cond"], g["uncond"], case["cfg"], case["steps"], case["eta"],
                          list(g["noises"]))
    assert info["evaluations"] == len(g["model_times"]) == case["steps"]
    assert torch.allclose(info["model_times"], g["model_times"], atol=1e-3)
    assert _rel(out, g["out"]) < 1e-6
    assert _rel(info["x_after_first_corrector"], g["x_after_first_corrector"]) < 1e-6


def test_inference_default_times_and_tau_window():
    """S = 25: model times 999.0, 959.04, ..., 39.96; tau = eta on steps 6..20 (t in [0.2, 0.8] on the float32 grid)."""
    g = torch.load(os.path.join(GOLD, "sa_s25.pt"))
    assert [round(v, 2) for v in g["model_times"][:2].tolist()] == [999.0, 959.04] and round(float(g["model_times"][-1]), 2) == 39.96
    p = so.plan(25, 1)
    assert [i for i, e in enumerate(p) if e["tau_c"]] == list(range(6, 21))
    assert [i + 1 for i, e in enumerate(p) if e["tau_p"]] == list(range(6, 21))
    p5 = so.plan(5, 1)                                                  # t = 0.8 falls just outside the float32 window
    assert [i for i, e in enumerate(p5) if e["tau_c"]] == [2, 3, 4] and p5[1]["tau_c"] == 0


def _solver(**kw):
    return sampler.SASolverSampler(lambda *a, **k: None, **kw)


@pytest.mark.parametrize("eta", [0, 1])
@pytest.mark.parametrize("steps", [2, 5, 10, 25, 33])
def test_product_plan_matches_oracle(steps, eta):
    plan, want = _solver().plan(steps, eta), so.plan(steps, eta)
    assert len(plan) == len(want) == steps
    for i, (p, w) in enumerate(zip(plan, want)):
        assert (p["has_corr"], p["order"], p["tau_c"], p["tau_p"]) == (w["has_corr"], w["order"], w["tau_c"], w["tau_p"]), i
        for k in PLAN_KEYS:
            assert abs(p[k] - w[k]) <= 1e-6 * max(1.0, abs(w[k])), (i, k, p[k], w[k])
    assert plan[-1]["pN"] == 0.0 and plan[-1]["p1"] == 0.0 and not plan[0]["has_corr"]


def test_signatures_match_the_reference():
    """Constructor and `.sample` take the reference's parameters in the reference's order; `cuda_graph` is an added
    keyword-only parameter in front of **kwargs, so every positional call and keyword of the reference still binds."""
    g = torch.load(os.path.join(GOLD, "sa_s25.pt"))
    assert list(inspect.signature(sampler.SASolverSampler.__init__).parameters) == g["init_params"]
    params = inspect.signature(sampler.SASolverSampler.sample).parameters
    assert [n for n, p in params.items() if p.kind != p.KEYWORD_ONLY] == g["sample_params"]
    assert [n for n, p in params.items() if p.kind == p.KEYWORD_ONLY] == ["cuda_graph"]


def test_sampler_rejects_cpu_tensors_and_too_few_steps():
    s = _solver(device="cuda")
    with pytest.raises(RuntimeError, match="no CPU path"):
        s.sample(S=5, batch_size=1, shape=(4, 8, 8), conditioning=torch.zeros(1, 1, 2, 2), x_T=torch.zeros(1, 4, 8, 8))
    with pytest.raises(RuntimeError, match="no CPU path"):
        _solver().sample(S=5, batch_size=1, shape=(4, 8, 8), conditioning=torch.zeros(1, 1, 2, 2))
    with pytest.raises(ValueError):
        s.sample(S=1, batch_size=1, shape=(4, 8, 8), conditioning=torch.zeros(1, 1, 2, 2))
    with pytest.raises(NotImplementedError):
        _solver(noise_schedule="squaredcos_cap_v2")


def test_sa_step_struct_matches_header_size():
    """Size check of PxaSaStepArgs against a compile of the header with gcc (as test_ctypes_structs_match_header_sizes)."""
    src = '#include <stdio.h>\n#include "pixart_sm100.h"\nint main(){printf("%zu\\n", sizeof(PxaSaStepArgs));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        size = int(subprocess.check_output([os.path.join(d, "s")]))
    assert size == ctypes.sizeof(lib.SaStepArgs)


def test_install_into_reference_repoints_sa_solver_sampler(monkeypatch):
    import pixart_sigma_b200
    pkg, model_pkg = types.ModuleType("diffusion"), types.ModuleType("diffusion.model")
    nets, builder = types.ModuleType("diffusion.model.nets"), types.ModuleType("diffusion.model.builder")
    builder.MODELS = types.SimpleNamespace(_module_dict={})
    pkg.model, model_pkg.nets, model_pkg.builder = model_pkg, nets, builder
    pkg.SASolverSampler = pkg.DPMS = object()
    for mod in (pkg, model_pkg, nets, builder):
        monkeypatch.setitem(sys.modules, mod.__name__, mod)
    assert pixart_sigma_b200.install_into_reference()
    assert pkg.SASolverSampler is pixart_sigma_b200.SASolverSampler and pkg.DPMS is pixart_sigma_b200.DPMS
