"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's SA-Solver sampling loop as `scripts/inference.py` drives it
(`SASolverSampler(model.forward_with_dpmsolver, device).sample(S=25, batch_size=n, shape, eta=1, conditioning,
unconditional_conditioning, unconditional_guidance_scale, model_kwargs)`, scripts/inference.py:119-133).  Only tests and
tools may import this module; the product (`pixart_sigma_b200/sampler.py`) must not.

Pinned against the unmodified reference (`diffusion/sa_sampler.py::SASolverSampler`, imported through oracle/refshim.py) by
`oracle/gen_golden_sa.py` -> `tests/golden/sa_*.pt`, checked in tests/test_sa_solver_cpu.py.

What is restated (file:line in the reference checkout):
  * alphas_cumprod = float32(cumprod(1 - linear betas))     diffusion/sa_sampler.py:19-22
  * NoiseScheduleVP('discrete', alphas_cumprod=...): float32 log-alpha table 0.5 log(alphas_cumprod), no lambda clipping,
    piecewise-linear look-ups                             diffusion/model/sa_solver.py:81-90,108-140,1099-1137
  * model_wrapper('noise', 'classifier-free'): t_input = (t - 1/N) * 1000, CFG batch [uncond ; cond], a single
    conditional evaluation when guidance_scale == 1 or uncond is None
                                                          diffusion/model/sa_solver.py:259-318
  * data prediction x0 = (x - sigma eps) / alpha            diffusion/model/sa_solver.py:377-386
  * tau(t) = eta if 0.2 <= t <= 0.8 else 0 on the float32 time grid
                                                          diffusion/sa_sampler.py:90
  * skip_type='time', skip_order=1: linspace(1, 1/N, S+1) diffusion/model/sa_solver.py:408-410
  * Lagrange x exponential-integral coefficients, data-prediction form
                                                          diffusion/model/sa_solver.py:449-560
  * predictor / corrector with the order-2 "few steps" term
                                                          diffusion/model/sa_solver.py:644-753
  * sample_few_steps, predictor_order=2, corrector_order=2, PEC, lower_order_final, last step tau = 0
                                                          diffusion/model/sa_solver.py:755-909
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence

import numpy as np
import torch

from oracle.dpm_oracle import DiscreteSchedule, linear_betas, toy_model  # noqa: F401  (toy_model re-exported for the tests)


class AlphasCumprodSchedule(DiscreteSchedule):
    """The DPM schedule's look-ups over the SA table: log(alpha) = 0.5 log(alphas_cumprod) in float32."""

    def __init__(self, diffusion_steps: int = 1000):
        alphas = 1.0 - torch.tensor(linear_betas(diffusion_steps))                      # float64
        alphas_cumprod = torch.cumprod(alphas, dim=0).to(torch.float32)
        self.log_alpha = (0.5 * torch.log(alphas_cumprod)).to(torch.float32)
        self.total_N = self.log_alpha.numel()
        self.t = torch.linspace(0., 1., self.total_N + 1)[1:].to(torch.float32)
        self.T = 1.0


def time_grid(sch: AlphasCumprodSchedule, steps: int) -> torch.Tensor:
    return torch.linspace(sch.T, 1. / sch.total_N, steps + 1)


def tau_of(t: torch.Tensor, eta):
    return eta if 0.2 <= t <= 0.8 else 0


def _exp_integral(order: int, start, end, tau):
    """int exp(x (1 + tau^2)) x^order dx over [start, end], orders 0 and 1 (sa_solver.py:449-471)."""
    k = 1 + tau ** 2
    end_c, start_c = k * end, k * start
    if order == 0:
        return torch.exp(end_c) * (1 - torch.exp(-(end_c - start_c))) / k
    return torch.exp(end_c) * ((end_c - 1) - (start_c - 1) * torch.exp(-(end_c - start_c))) / (k ** 2)


def _gradient_coefficients(order: int, lam_start, lam_end, lams: Sequence, tau) -> List:
    """Lagrange basis through `lams` integrated against the exponential weight (sa_solver.py:478-560), orders 1 and 2."""
    if order == 1:
        lagrange = [[1]]
    else:
        l0, l1 = lams
        lagrange = [[1 / (l0 - l1), -l1 / (l0 - l1)], [1 / (l1 - l0), -l0 / (l1 - l0)]]
    out = []
    for i in range(order):
        c = 0
        for j in range(order):
            c += lagrange[i][j] * _exp_integral(order - 1 - j, lam_start, lam_end, tau)
        out.append(c)
    return out


def update_coefficients(sch: AlphasCumprodSchedule, order: int, tau, t_prev: Sequence[torch.Tensor], t: torch.Tensor,
                        corrector: bool):
    """x_new = A x + g[0] m[-1] + g[1] m[-2] + N noise (g[1] = 0 at order 1), every scalar a float32 (1,) tensor computed as
    adams_bashforth_update_few_steps (corrector=False) / adams_moulton_update_few_steps (corrector=True) compute it."""
    sigma_t, lam_t = sch.sigma(t), sch.lam(t)
    sigma_prev, lam_prev = sch.sigma(t_prev[-1]), sch.lam(t_prev[-1])
    h = lam_t - lam_prev
    ts = (list(t_prev) + [t]) if corrector else list(t_prev)
    lams = [sch.lam(ts[-(i + 1)]) for i in range(order)]
    g = _gradient_coefficients(order, lam_prev, lam_t, lams, tau)
    if order == 2:
        k = 1 + tau ** 2
        if corrector:
            extra = 1.0 * torch.exp(k * lam_t) * (h / 2 - (h * k - 1 + torch.exp(k * (-h))) / (k ** 2 * h))
        else:
            extra = 1.0 * torch.exp(k * lam_t) * (h ** 2 / 2 - (h * k - 1 + torch.exp(k * (-h))) / (k ** 2)) / (
                lam_prev - sch.lam(t_prev[-2]))
        g[0] += extra
        g[1] -= extra
    coef = [(1 + tau ** 2) * sigma_t * torch.exp(- tau ** 2 * lam_t) * gi for gi in g]
    A = torch.exp(-tau ** 2 * h) * (sigma_t / sigma_prev)
    N = sigma_t * torch.sqrt(1 - torch.exp(-2 * tau ** 2 * h))
    return A, coef, N


def _apply(A, coef, N, x, models, noise):
    grad = torch.zeros_like(x)
    for i, c in enumerate(coef):
        grad += c * models[-(i + 1)]
    return A * x + grad + N * noise


def plan(steps: int, eta, sch: Optional[AlphasCumprodSchedule] = None) -> List[dict]:
    """Per denoiser evaluation i (at ts[i]): the scalars of one fused SA step (the corrector of step i, then the predictor of
    step i + 1), as floats.  Each comes out of the same float32 operations `sample` applies to the tensors."""
    sch = sch or AlphasCumprodSchedule()
    ts = time_grid(sch, steps)
    out = []
    for i in range(steps):
        t = ts[i]
        e = dict(t_input=float((t - 1. / sch.total_N) * 1000.), sigma=float(sch.sigma(t)),
                 inv_alpha=float(1. / sch.alpha(t)), has_corr=i >= 1, tau_c=0, tau_p=0)
        if i >= 1:
            e["tau_c"] = tau_of(t, eta)
            A, (c0, c1), N = update_coefficients(sch, 2, e["tau_c"], [ts[j] for j in range(max(0, i - 2), i)], t, True)
            e.update(cA=float(A), c0=float(c0), c1=float(c1), cN=float(N))
        else:
            e.update(cA=0., c0=0., c1=0., cN=0.)
        step = i + 1
        order = 1 if step == 1 or step == steps else 2
        e["tau_p"] = 0 if step == steps else tau_of(ts[step], eta)
        A, coef, N = update_coefficients(sch, order, e["tau_p"], [ts[j] for j in range(max(0, i - 1), i + 1)], ts[step], False)
        e.update(pA=float(A), p0=float(coef[0]), p1=float(coef[1]) if order == 2 else 0., pN=float(N), order=order)
        out.append(e)
    return out


def sample(model: Callable, x_T: torch.Tensor, condition: torch.Tensor, uncondition: Optional[torch.Tensor], cfg_scale: float,
           steps: int, eta, noises: Sequence[torch.Tensor], model_kwargs: Optional[dict] = None):
    """`model(x, t_input, cond, **model_kwargs) -> eps`; `noises`: the S + 1 draws of the reference loop (draw 0 unused).
    Returns (x, info) with info = dict(model_times, x_after_first_corrector, evaluations)."""
    assert steps >= 2 and len(noises) == steps + 1
    model_kwargs = model_kwargs or {}
    sch = AlphasCumprodSchedule()
    ts = time_grid(sch, steps)
    guided = not (cfg_scale == 1. or uncondition is None)
    seen: List[float] = []

    def data_pred(x, t):
        t_in = (t.expand(x.shape[0]) - 1. / sch.total_N) * 1000.
        if guided:
            out = model(torch.cat([x] * 2), torch.cat([t_in] * 2), torch.cat([uncondition, condition]), **model_kwargs)
            eu, ec = out.chunk(2)
            eps = eu + cfg_scale * (ec - eu)
        else:
            eps = model(x, t_in, condition, **model_kwargs)
        seen.append(float(t_in[0]))
        return (x - sch.sigma(t) * eps) / sch.alpha(t)

    x = x_T
    models = [data_pred(x, ts[0])]
    t_prev = [ts[0]]
    first_corr = None
    for step in range(1, steps + 1):
        t = ts[step]
        noise = noises[step]
        last = step == steps
        p_order = 1 if step == 1 or last else 2
        A, coef, N = update_coefficients(sch, p_order, 0 if last else tau_of(t, eta), t_prev, t, False)
        x_p = _apply(A, coef, N, x, models, noise)
        if last:
            x = x_p
            break
        models.append(data_pred(x_p, t))
        A, coef, N = update_coefficients(sch, 2, tau_of(t, eta), t_prev, t, True)
        x = _apply(A, coef, N, x, models, noise)
        if first_corr is None:
            first_corr = x
        t_prev.append(t)
        models = models[-2:]
    return x, dict(model_times=torch.tensor(seen), x_after_first_corrector=first_corr, evaluations=len(seen))
