"""GPU tests (-m gpu) of the SA-Solver sampler: the fused step kernel (pxa_sa_solver_step) against its fp32 formula, and the
sampling loop of pixart_sigma_b200/sampler.py::SASolverSampler against the reference fixtures (oracle/gen_golden_sa.py), the
oracle restatement (oracle/sa_oracle.py) and the reference's consumption of the CUDA generator.

Tolerances: step kernel vs the fp32 formula 1e-6 (each operation rounded as in the formula; only the reciprocal of alpha
differs); loop with the toy denoiser vs the reference fixture 1e-5 (the toy loop amplifies an input perturbation about 2x);
loop around the sm_100a PixArtMS vs the oracle loop around the oracle forward 2e-2 (5 denoiser evaluations at the model's
~3e-3 each, amplified by the solver's 1/alpha factors -- the bar of the DPM-Solver++ loop test)."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pixart_oracle as po          # noqa: E402
from oracle import sa_oracle as so              # noqa: E402
from oracle.gen_golden_sa import CASES          # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden")
DEV = "cuda"

if torch.cuda.is_available():
    from pixart_sigma_b200 import PixArtMS, lib, sampler


def _rel(a, b):
    return float((a.float().cpu() - b.float().cpu()).norm() / b.float().cpu().norm())


def _replay(noises):
    """A `_draw` that hands out the recorded noises in order, as device-to-device copies (so a graph capture keeps them)."""
    seq = [z.to(DEV) for z in noises]
    calls = []

    def draw(buf):
        buf.copy_(seq[len(calls)])
        calls.append(1)
    return draw, calls


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("learn_sigma_view", [False, True])
@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("has_corr", [False, True])
@pytest.mark.parametrize("p1", [0.0, -0.37])
def test_step_kernel_matches_formula(dtype, learn_sigma_view, guided, has_corr, p1):
    g = torch.Generator().manual_seed(7)
    n, h, w = 3, 24, 20
    rows = 2 * n if guided else n
    full = torch.randn(rows, 8 if learn_sigma_view else 4, h, w, generator=g).to(dtype)
    out = full[:, :4]                                           # the view forward_with_dpmsolver returns for learn-sigma
    x, xp, prev, nz, nn = (torch.randn(n, 4, h, w, generator=g) for _ in range(5))
    k = dict(cfg_scale=4.5, sigma=0.83, inv_alpha=1.0 / 0.557, has_corr=has_corr, cA=0.71, c0=0.52, c1=-0.11, cN=0.33,
             pA=0.64, p0=0.41, p1=p1, pN=0.29)
    o = out.float()
    eps = o[:n] + k["cfg_scale"] * (o[n:] - o[:n]) if guided else o
    x0 = (xp - k["sigma"] * eps) * k["inv_alpha"]
    xc = (k["cA"] * x + (k["c0"] * x0 + k["c1"] * prev)) + k["cN"] * nz if has_corr else xp
    want = (k["pA"] * xc + (k["p0"] * x0 + k["p1"] * prev)) + k["pN"] * nn
    dx, dxp, dprev, dnz, dnn = (t.to(DEV) for t in (x, xp, prev, nz, nn))
    lib.sa_solver_step(full.to(DEV)[:, :4], dx, dxp, dprev, dnz, dnn, guided=guided, **k)
    assert _rel(dxp, want) < 1e-6
    assert _rel(dx, xc) < 1e-6
    assert _rel(dprev, x0) < 1e-6


@pytest.mark.parametrize("name", sorted(CASES))
def test_loop_with_toy_denoiser_matches_reference_fixture(name):
    case, g = CASES[name], torch.load(os.path.join(GOLD, name + ".pt"))
    solver = sampler.SASolverSampler(so.toy_model, device=DEV)
    kw = dict(S=case["steps"], batch_size=case["n"], shape=(4,) + case["hw"], conditioning=g["cond"].to(DEV), eta=case["eta"],
              x_T=g["x_T"].to(DEV), unconditional_guidance_scale=case["cfg"],
              unconditional_conditioning=None if g["uncond"] is None else g["uncond"].to(DEV), model_kwargs={})
    solver._draw, calls = _replay(g["noises"])
    out, second = solver.sample(**kw)
    assert second is None and out.dtype == torch.float32 and len(calls) == case["steps"] + 1
    assert _rel(out, g["out"]) < 1e-5
    solver._draw, calls = _replay(g["noises"])
    graphed, _ = solver.sample(**kw, cuda_graph=True)                   # capture + first replay
    assert len(calls) == case["steps"] + 1 and _rel(graphed, g["out"]) < 1e-5
    again, _ = solver.sample(**kw, cuda_graph=True)                     # replay of the cached graph
    assert len(calls) == case["steps"] + 1 and torch.equal(graphed, again)


def test_seeded_run_consumes_the_generator_like_the_reference():
    """x_T None: the sampler draws x_T and then S + 1 noises of x_T's shape from the default CUDA generator, exactly what
    `torch.randn(size, device)` followed by the loop's S + 1 `torch.randn_like(x)` draw in the reference."""
    case = CASES["sa_s5"]
    g = torch.load(os.path.join(GOLD, "sa_s5.pt"))
    n, (h, w), S = 2, case["hw"], case["steps"]
    cond, uncond = g["cond"].repeat(n, 1, 1, 1), g["uncond"].repeat(n, 1, 1, 1)
    solver = sampler.SASolverSampler(so.toy_model, device=DEV)
    kw = dict(S=S, batch_size=n, shape=(4, h, w), conditioning=cond.to(DEV), eta=1, unconditional_guidance_scale=4.5,
              unconditional_conditioning=uncond.to(DEV), model_kwargs={})
    torch.cuda.manual_seed(2024)
    out, _ = solver.sample(**kw)
    eager_state = torch.cuda.get_rng_state()
    torch.cuda.manual_seed(2024)
    x_T = torch.randn((n, 4, h, w), device=DEV)
    noises = [torch.randn_like(x_T) for _ in range(S + 1)]
    after = torch.cuda.get_rng_state()
    assert torch.equal(eager_state, after)
    want, _ = so.sample(so.toy_model, x_T.cpu(), cond, uncond, 4.5, S, 1, [z.cpu() for z in noises])
    assert _rel(out, want) < 1e-5
    torch.cuda.manual_seed(2024)
    graphed, _ = solver.sample(**kw, cuda_graph=True)
    assert torch.equal(torch.cuda.get_rng_state(), after)              # same generator position as the reference's draws
    assert float((graphed - out).abs().max()) <= 1e-6
    again, _ = solver.sample(**kw, cuda_graph=True)                    # no reseed: fresh x_T and noise
    assert not torch.equal(again, graphed)


def test_loop_around_the_sm100_model_matches_oracle_loop():
    """5-step eta = 1 CFG sampling of a depth-2 PixArtMS at 256px (latent 32x32) on the sm_100a kernels vs the oracle loop
    around the fp32 oracle forward on the same bf16-rounded weights and the same noises."""
    cfg = po.OracleConfig(depth=2, input_size=32, pe_interpolation=0.5)
    sd = {k: v.to(torch.bfloat16).float() for k, v in po.synthetic_state_dict(cfg, seed=0).items()}
    z, _, y, mask = po.synthetic_inputs(cfg, 1, (32, 32), seed=5, lens=[77])
    null_y = po.synthetic_inputs(cfg, 1, (32, 32), seed=6)[2]
    y, null_y = y.to(torch.bfloat16).float(), null_y.to(torch.bfloat16).float()
    with torch.device(DEV):
        m = PixArtMS(depth=2, input_size=32, pe_interpolation=0.5, model_max_length=300)
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected and missing == ["pos_embed"]
    m = m.to(torch.bfloat16).eval()
    kw = dict(data_info=None, mask=mask.to(DEV))
    S = 5
    noises = list(torch.randn(S + 1, *z.shape, generator=torch.Generator().manual_seed(11)))
    solver = sampler.SASolverSampler(m.forward_with_dpmsolver, device=DEV)
    args = dict(S=S, batch_size=1, shape=(4, 32, 32), conditioning=y.to(DEV), eta=1, x_T=z.to(DEV),
                unconditional_guidance_scale=4.5, unconditional_conditioning=null_y.to(DEV), model_kwargs=kw)
    with torch.no_grad():
        t0 = torch.full((2,), 999.0, device=DEV)
        m.forward_with_dpmsolver(torch.cat([z, z]).to(DEV), t0, torch.cat([null_y, y]).to(DEV), **kw)   # lazy inits
        n0 = lib.launch_count()
        m.forward_with_dpmsolver(torch.cat([z, z]).to(DEV), t0, torch.cat([null_y, y]).to(DEV), **kw)
        per_forward = lib.launch_count() - n0
    solver._draw, _ = _replay(noises)
    n0 = lib.launch_count()
    out, _ = solver.sample(**args)
    assert per_forward >= 2 * 11 and lib.launch_count() - n0 == S * (per_forward + 1)   # + one step kernel per evaluation

    def oracle_model(x, t, c, **kwargs):
        return po.forward_with_dpmsolver(sd, cfg, x, t, c, data_info=None, mask=mask)
    want, _ = so.sample(oracle_model, z, y, null_y, 4.5, S, 1, noises)
    err = _rel(out, want)
    assert err < 2e-2, f"SA-Solver 5-step eta=1 loop, depth 2, 256px: rel_err vs the oracle loop = {err:.3e}"
    solver._draw, _ = _replay(noises)
    graphed, _ = solver.sample(**args, cuda_graph=True)
    assert _rel(graphed, out) < 1e-5
