"""TEST INFRASTRUCTURE ONLY -- generate tests/golden/sa_*.pt by running the UNMODIFIED reference SA-Solver sampler
(`diffusion.SASolverSampler`, imported through oracle/refshim.py) on seeded inputs with the deterministic toy denoiser of
oracle/dpm_oracle.py.  Needs a reference checkout (see oracle/refshim.py):  python oracle/gen_golden_sa.py

The wrapper moves its `alphas_cumprod` buffer to CUDA unconditionally (diffusion/sa_sampler.py:24-28); the script replaces
that method on the class for its own run so the buffer stays on the CPU.  `torch.randn_like` is wrapped to record the S + 1
noise draws of the loop, and the predictor to record the state after the first corrector (its `x` at the second call).
"""
import inspect
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import dpm_oracle as do               # noqa: E402
from oracle.refshim import install_reference_shims  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
CASES = {"sa_s25": dict(steps=25, eta=1, cfg=4.5, n=2, hw=(8, 12), uncond=True),       # scripts/inference.py:119-133
         "sa_s5": dict(steps=5, eta=1, cfg=4.5, n=1, hw=(8, 8), uncond=True),          # tau window: t = 0.6, 0.4, 0.2
         "sa_s2_eta0": dict(steps=2, eta=0, cfg=4.5, n=1, hw=(8, 8), uncond=True),     # the minimum, deterministic
         "sa_s10_nouncond": dict(steps=10, eta=1, cfg=4.5, n=2, hw=(8, 8), uncond=False),
         "sa_s10_cfg1": dict(steps=10, eta=1, cfg=1.0, n=2, hw=(8, 8), uncond=True)}


def inputs(case, seed=0):
    g = torch.Generator().manual_seed(seed)
    n, (h, w) = case["n"], case["hw"]
    x_T = torch.randn(n, 4, h, w, generator=g)
    cond = torch.randn(n, 1, 6, 8, generator=g) * 0.5
    uncond = (torch.randn(1, 1, 6, 8, generator=g) * 0.5).repeat(n, 1, 1, 1)
    return x_T, cond, (uncond if case["uncond"] else None)


def main():
    install_reference_shims()
    import tqdm as _tqdm  # noqa: F401  (the reference's loop wraps its ranges in tqdm)
    from diffusion import SASolverSampler
    from diffusion.model import sa_solver
    SASolverSampler.register_buffer = lambda self, name, attr: setattr(self, name, attr)
    os.makedirs(OUT, exist_ok=True)
    randn_like, predictor = torch.randn_like, sa_solver.SASolver.adams_bashforth_update_few_steps
    for name, case in CASES.items():
        x_T, cond, uncond = inputs(case)
        draws, seen, pred_x = [], [], []

        def spy(x, t, c, **kw):
            seen.append(float(t[0]))
            return do.toy_model(x, t, c, **kw)

        def recording_randn_like(x, *a, **k):
            v = randn_like(x, *a, **k)
            draws.append(v.clone())
            return v

        def recording_predictor(self, order, x, *a, **k):
            pred_x.append(x.clone())
            return predictor(self, order, x, *a, **k)

        torch.manual_seed(1234)
        torch.randn_like, sa_solver.SASolver.adams_bashforth_update_few_steps = recording_randn_like, recording_predictor
        try:
            sampler = SASolverSampler(spy, device="cpu")
            out, second = sampler.sample(S=case["steps"], batch_size=case["n"], shape=(4,) + case["hw"], conditioning=cond,
                                         eta=case["eta"], x_T=x_T.clone(), unconditional_guidance_scale=case["cfg"],
                                         unconditional_conditioning=uncond, model_kwargs={}, verbose=False)
        finally:
            torch.randn_like, sa_solver.SASolver.adams_bashforth_update_few_steps = randn_like, predictor
        assert second is None
        torch.save(dict(case=case, x_T=x_T, cond=cond, uncond=uncond, noises=torch.stack(draws), model_times=torch.tensor(seen),
                        x_after_first_corrector=pred_x[1], out=out,
                        sample_params=list(inspect.signature(SASolverSampler.sample).parameters),
                        init_params=list(inspect.signature(SASolverSampler.__init__).parameters)),
                   os.path.join(OUT, name + ".pt"))
        print(name, tuple(out.shape), len(seen), "evaluations", len(draws), "draws, times", [round(v, 2) for v in seen[:3]], "...")


if __name__ == "__main__":
    main()
