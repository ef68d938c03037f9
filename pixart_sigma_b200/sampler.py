"""B200-native drivers of the DPM-Solver++ and SA-Solver sampling loops around the denoiser hot path (SURVEY.md §8f.1).

Mirrors the reference's `diffusion.DPMS(...)` factory and `DPM_Solver.sample(...)` as `scripts/inference.py:102-118` uses
them (`diffusion/dpm_solver.py:6-35`, `diffusion/model/dpm_solver.py:1069-1241`): same call signature, same result, for
the configuration the reference ships (noise-prediction model, classifier-free guidance, linear discrete schedule,
`algorithm_type="dpmsolver++"`, `method="multistep"`, `order<=2`, `skip_type="time_uniform"`).  Other options raise
`NotImplementedError` instead of silently taking a different path.

What is different from the reference loop:
  * all schedule look-ups (the reference's `interpolate_fn` sorts a 1001-element array on the GPU for every alpha /
    sigma / lambda it needs, ~10 tiny kernels + syncs per step) are done ONCE on the host: per step five scalars;
  * CFG combine, data prediction and the first / second-order multistep update are ONE elementwise sm_100a kernel per
    step (`pxa_dpm_solver_pp_step`, include/pixart_sm100.h) instead of ~25 PyTorch elementwise launches;
  * `cuda_graph=True` captures the whole `steps`-step loop (denoiser launches included) into one CUDA graph.
There is no CPU path: inputs must live on an sm_100 device.

`SASolverSampler` does the same for the reference's `diffusion.SASolverSampler` (`--sampling_algo sa-solver`,
scripts/inference.py:119-133) with one fused predictor-corrector kernel per denoiser evaluation (`pxa_sa_solver_step`).
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import numpy as np
import torch

from . import lib

__all__ = ["DPMS", "DPMSolverPP", "SASolverSampler"]


class _DiscreteVPSchedule:
    """log(alpha) of the discrete linear-beta VP schedule at t_i = i/N (float32 table, piecewise-linear look-up with the
    outermost segments extended), as `NoiseScheduleVP('discrete', betas=linear)` defines it
    (diffusion/model/dpm_solver.py:97-106,127-155; betas: diffusion/model/gaussian_diffusion.py:82,107-116)."""

    def __init__(self, diffusion_steps: int = 1000, clipped_lambda: float = -5.1):
        scale = 1000 / diffusion_steps
        betas = np.linspace(scale * 0.0001, scale * 0.02, diffusion_steps, dtype=np.float64)
        log_alphas = 0.5 * torch.log(1 - torch.from_numpy(betas)).cumsum(dim=0)
        lambs = log_alphas - 0.5 * torch.log(1. - torch.exp(2. * log_alphas))
        drop = int(torch.searchsorted(torch.flip(lambs, [0]), torch.tensor(clipped_lambda, dtype=lambs.dtype)))
        if drop > 0:                       # log-SNR clipped near t = T (a no-op for the linear schedule)
            log_alphas = log_alphas[:-drop]
        self.log_alpha = log_alphas.to(torch.float32)
        self.total_N = self.log_alpha.numel()
        self.t = torch.linspace(0., 1., self.total_N + 1)[1:].to(torch.float32)
        self.T = 1.0

    def log_alpha_at(self, t: torch.Tensor) -> torch.Tensor:
        t = t.reshape(-1).to(torch.float32)
        seg = (torch.searchsorted(self.t, t.contiguous()) - 1).clamp(0, self.total_N - 2)
        t0, t1, y0, y1 = self.t[seg], self.t[seg + 1], self.log_alpha[seg], self.log_alpha[seg + 1]
        return y0 + (t - t0) * (y1 - y0) / (t1 - t0)

    def alpha(self, t):
        return torch.exp(self.log_alpha_at(t))

    def sigma(self, t):
        return torch.sqrt(1. - torch.exp(2. * self.log_alpha_at(t)))

    def lam(self, t):
        la = self.log_alpha_at(t)
        return la - 0.5 * torch.log(1. - torch.exp(2. * la))


class _AlphasCumprodSchedule(_DiscreteVPSchedule):
    """The same look-ups over the table `NoiseScheduleVP('discrete', alphas_cumprod=...)` builds for the SA-Solver wrapper:
    log(alpha) = 0.5 log(alphas_cumprod) with alphas_cumprod = float32(cumprod(1 - linear betas)), the logarithm taken in
    float32, no log-SNR clipping (diffusion/sa_sampler.py:19-22, diffusion/model/sa_solver.py:81-90)."""

    def __init__(self, diffusion_steps: int = 1000):
        scale = 1000 / diffusion_steps
        betas = np.linspace(scale * 0.0001, scale * 0.02, diffusion_steps, dtype=np.float64)
        alphas_cumprod = torch.cumprod(1.0 - torch.from_numpy(betas), dim=0).to(torch.float32)
        self.log_alpha = 0.5 * torch.log(alphas_cumprod)
        self.total_N = self.log_alpha.numel()
        self.t = torch.linspace(0., 1., self.total_N + 1)[1:].to(torch.float32)
        self.T = 1.0


def _captured_model_key(model: Callable, params: List[torch.Tensor], model_kwargs: dict) -> tuple:
    """What a captured denoiser call depends on beyond its inputs: the model_kwargs tensors (captured by address) and, when the
    forward keeps derived copies of its weights (stacked kv_linear weights, fused-LN tables) that a replay cannot refresh, the
    parameters' versions."""
    kw_id = tuple(sorted((k, (v.data_ptr(), tuple(v.shape)) if isinstance(v, torch.Tensor) else repr(v))
                         for k, v in (model_kwargs or {}).items()))
    owner = getattr(model, "__self__", model)
    derived = getattr(owner, "_kv_batch", None) is not None or getattr(owner, "_ln_fusion", None) is not None
    wkey = (sum(p._version for p in params), params[0].data_ptr()) if (params and derived) else None
    return kw_id, wkey


class DPMSolverPP:
    """Multistep DPM-Solver++ (order 1 / 2) with classifier-free guidance; see the module docstring."""

    def __init__(self, model: Callable, condition: torch.Tensor, uncondition: Optional[torch.Tensor], cfg_scale: float,
                 model_kwargs: Optional[dict] = None, diffusion_steps: int = 1000):
        self.model = model
        self.condition = condition
        self.uncondition = uncondition
        self.cfg_scale = float(cfg_scale)
        self.model_kwargs = dict(model_kwargs or {})
        self.schedule = _DiscreteVPSchedule(diffusion_steps)
        self._graphs: Dict[tuple, tuple] = {}
        self._cfg_cond: Optional[torch.Tensor] = None          # cat([uncondition, condition]), built once
        owner = getattr(model, "__self__", model)              # the nn.Module behind a bound forward_with_dpmsolver
        self._params = list(owner.parameters()) if isinstance(owner, torch.nn.Module) else []

    # ---- host side: everything that does not depend on the latents
    def plan(self, steps: int, order: int = 2, t_start: Optional[float] = None, t_end: Optional[float] = None,
             lower_order_final: bool = True) -> List[dict]:
        """Per update i (time ts[i] -> ts[i+1]): the model-input time and the five scalars of pxa_dpm_solver_pp_step."""
        sch = self.schedule
        t_0 = 1. / sch.total_N if t_end is None else t_end
        t_T = sch.T if t_start is None else t_start
        assert t_0 > 0 and t_T > 0, "time range must be positive (discrete-time DPMs: [1/N, 1])"
        assert steps >= order
        ts = torch.linspace(t_T, t_0, steps + 1)                       # time_uniform (dpm_solver.py:475-476)
        plan = []
        for i in range(steps):
            s, t = ts[i:i + 1], ts[i + 1:i + 2]
            step = i + 1
            step_order = 1 if step < order else (min(order, steps + 1 - step) if lower_order_final else order)
            h = sch.lam(t) - sch.lam(s)
            b = torch.exp(sch.log_alpha_at(t)) * torch.expm1(-h)        # alpha_t * phi_1
            c = torch.zeros_like(b)
            if step_order == 2:
                r0 = (sch.lam(s) - sch.lam(ts[i - 1:i])) / h
                c = 0.5 * b * (1. / r0)
            plan.append(dict(t_input=float((s - 1. / sch.total_N) * 1000.), sigma_s=float(sch.sigma(s)),
                             alpha_s=float(sch.alpha(s)), a=float(sch.sigma(t) / sch.sigma(s)), b=float(b), c=float(c),
                             order=step_order))
        return plan

    # ---- device side
    def _run(self, x: torch.Tensor, x0_prev: torch.Tensor, plan: List[dict], t_dev: List[torch.Tensor], cond: torch.Tensor,
             inter: Optional[list]) -> torch.Tensor:
        n = x.shape[0]
        guided = self.uncondition is not None and self.cfg_scale != 1.
        for st, t_in in zip(plan, t_dev):
            if guided:
                out = self.model(torch.cat([x, x]), t_in, cond, **self.model_kwargs)
            else:                                   # reference: a single conditional evaluation (dpm_solver.py:327-328)
                out = self.model(x, t_in[:n], cond, **self.model_kwargs)
                out = torch.cat([out, out])
            if out.dtype not in (torch.float32, torch.bfloat16):
                out = out.float()
            if not (out.stride(3) == 1 and out.stride(2) == out.shape[3] and out.stride(1) == out.shape[2] * out.shape[3]):
                out = out.contiguous()
            lib.dpm_solver_pp_step(out, x, x0_prev, cfg_scale=self.cfg_scale if guided else 1.0, sigma_s=st["sigma_s"],
                                   alpha_s=st["alpha_s"], a=st["a"], b=st["b"], c=st["c"])
            if inter is not None:
                inter.append(x.clone())
        return x

    @torch.no_grad()
    def sample(self, x: torch.Tensor, steps: int = 20, t_start: Optional[float] = None, t_end: Optional[float] = None,
               order: int = 2, skip_type: str = "time_uniform", method: str = "multistep", lower_order_final: bool = True,
               denoise_to_zero: bool = False, solver_type: str = "dpmsolver", atol: float = 0.0078, rtol: float = 0.05,
               return_intermediate: bool = False, cuda_graph: bool = False):
        if method != "multistep" or skip_type != "time_uniform" or solver_type != "dpmsolver" or denoise_to_zero or order > 2:
            raise NotImplementedError("only method='multistep', skip_type='time_uniform', solver_type='dpmsolver', "
                                      "order <= 2, denoise_to_zero=False (the configuration scripts/inference.py uses)")
        if not x.is_cuda:
            raise RuntimeError("pixart_sigma_b200.sampler has no CPU path: x must be a CUDA tensor")
        if x.dim() != 4 or x.shape[1] != 4 or (x.shape[2] * x.shape[3]) % 4:
            raise ValueError("x must be (n, 4, h, w) latents with h*w a multiple of 4")
        plan = self.plan(steps, order, t_start, t_end, lower_order_final)
        n = x.shape[0]
        guided = self.uncondition is not None and self.cfg_scale != 1.
        if guided and self._cfg_cond is None:
            self._cfg_cond = torch.cat([self.uncondition, self.condition])    # [uncond ; cond] (dpm_solver.py:330)
        cond = self._cfg_cond if guided else self.condition
        t_dev = [torch.full((2 * n,), st["t_input"], dtype=torch.float32, device=x.device) for st in plan]
        if cuda_graph and not return_intermediate:
            return self._sample_graphed(x, plan, t_dev, cond)
        xs = x.to(torch.float32).contiguous().clone()
        x0_prev = torch.empty_like(xs)
        inter = [] if return_intermediate else None
        out = self._run(xs, x0_prev, plan, t_dev, cond, inter)
        out = out.to(x.dtype)
        return (out, inter) if return_intermediate else out

    def _sample_graphed(self, x, plan, t_dev, cond):
        # every per-step scalar (sigma_s, alpha_s, a, b, c), the step orders and t_input are baked into the captured kernel
        # arguments, and `cond` / model_kwargs tensors into the captured forward: all of them are part of the key
        key = (tuple(x.shape), x.device.index, float(self.cfg_scale), cond.data_ptr(), tuple(cond.shape),
               _captured_model_key(self.model, self._params, self.model_kwargs),
               tuple((st["t_input"], st["sigma_s"], st["alpha_s"], st["a"], st["b"], st["c"], st.get("order")) for st in plan))
        if key not in self._graphs:
            x_static = x.to(torch.float32).contiguous().clone()
            x0_prev = torch.empty_like(x_static)
            z_in = torch.empty_like(x_static)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                      # warm-up outside capture (lazy inits, tensor maps)
                self._run(x_static, x0_prev, plan[:2], t_dev[:2], cond, None)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                x_static.copy_(z_in)
                self._run(x_static, x0_prev, plan, t_dev, cond, None)
            self._graphs[key] = (graph, z_in, x_static, t_dev, cond)
        graph, z_in, x_static = self._graphs[key][:3]
        z_in.copy_(x)
        graph.replay()
        return x_static.to(x.dtype).clone()


def DPMS(model: Callable, condition: torch.Tensor, uncondition: Optional[torch.Tensor], cfg_scale: float,
         model_type: str = "noise", noise_schedule: str = "linear", guidance_type: str = "classifier-free",
         model_kwargs: Optional[dict] = None, diffusion_steps: int = 1000) -> DPMSolverPP:
    """Same signature as the reference factory (`diffusion/dpm_solver.py:6-35`); returns an object with `.sample(...)`."""
    if model_type != "noise" or noise_schedule != "linear" or guidance_type != "classifier-free":
        raise NotImplementedError("only model_type='noise', noise_schedule='linear', guidance_type='classifier-free' "
                                  "(what scripts/inference.py uses)")
    return DPMSolverPP(model, condition, uncondition, cfg_scale, model_kwargs, diffusion_steps)


# ------------------------------------------------------------------------------------------------- SA-Solver
def _exp_integral(order: int, start, end, tau):
    """int_start^end exp(x (1 + tau^2)) x^order dx for order 0 / 1 (diffusion/model/sa_solver.py:449-471)."""
    k = 1 + tau ** 2
    end_c, start_c = k * end, k * start
    if order == 0:
        return torch.exp(end_c) * (1 - torch.exp(-(end_c - start_c))) / k
    return torch.exp(end_c) * ((end_c - 1) - (start_c - 1) * torch.exp(-(end_c - start_c))) / (k ** 2)


def _sa_update(sch: _DiscreteVPSchedule, order: int, tau, t_prev: List[torch.Tensor], t: torch.Tensor, corrector: bool):
    """(A, [g0, g1], N) of x_new = A x + g0 m[-1] + g1 m[-2] + N noise for the data-prediction SA predictor (corrector=False)
    or corrector of `order` 1 / 2 with the "few steps" term (diffusion/model/sa_solver.py:478-560,644-753), as float32 (1,)
    tensors computed by the reference's operations in the reference's order."""
    sigma_t, lam_t = sch.sigma(t), sch.lam(t)
    lam_prev = sch.lam(t_prev[-1])
    h = lam_t - lam_prev
    nodes = (t_prev + [t]) if corrector else t_prev
    if order == 1:
        lagrange = [[1]]
    else:
        l0, l1 = sch.lam(nodes[-1]), sch.lam(nodes[-2])
        lagrange = [[1 / (l0 - l1), -l1 / (l0 - l1)], [1 / (l1 - l0), -l0 / (l1 - l0)]]
    g = []
    for i in range(order):
        c = 0
        for j in range(order):
            c += lagrange[i][j] * _exp_integral(order - 1 - j, lam_prev, lam_t, tau)
        g.append(c)
    if order == 2:
        k = 1 + tau ** 2
        if corrector:
            extra = 1.0 * torch.exp(k * lam_t) * (h / 2 - (h * k - 1 + torch.exp(k * (-h))) / (k ** 2 * h))
        else:
            extra = 1.0 * torch.exp(k * lam_t) * (h ** 2 / 2 - (h * k - 1 + torch.exp(k * (-h))) / (k ** 2)) / (
                lam_prev - sch.lam(t_prev[-2]))
        g = [g[0] + extra, g[1] - extra]
    g = [(1 + tau ** 2) * sigma_t * torch.exp(- tau ** 2 * lam_t) * gi for gi in g]
    A = torch.exp(-tau ** 2 * h) * (sigma_t / sch.sigma(t_prev[-1]))
    N = sigma_t * torch.sqrt(1 - torch.exp(-2 * tau ** 2 * h))
    return A, g, N


class SASolverSampler:
    """The SA-Solver sampler of `diffusion.SASolverSampler` (diffusion/sa_sampler.py) on the sm_100a step kernel.

    Same constructor and `.sample(...)` signature and the same result as the reference wrapper, which always runs
    `SASolver(algorithm_type="data_prediction").sample(mode='few_steps', skip_type='time', skip_order=1, predictor_order=2,
    corrector_order=2, pc_mode='PEC', tau=lambda t: eta if 0.2 <= t <= 0.8 else 0)` around the noise-prediction model with
    classifier-free guidance.  The loop makes S denoiser evaluations and S + 1 standard-normal draws (the first one unused,
    the last one scaled by tau = 0), in the reference's order from the default CUDA generator, so a seeded run consumes the
    generator as the reference would.

    What is different from the reference loop: every schedule look-up and coefficient (each an `interpolate_fn` that sorts a
    1001-element array on the GPU in the reference, ~25-30 per step, plus a host sync for tau(t)) is computed once on the
    host by `plan`; the CFG combine, data prediction, corrector and next predictor are ONE elementwise kernel per evaluation
    (`pxa_sa_solver_step`, include/pixart_sm100.h); `cuda_graph=True` captures the noise draws and every denoiser and step
    launch of the loop into one CUDA graph.  There is no CPU path."""

    def __init__(self, model: Callable, noise_schedule="linear", diffusion_steps=1000, device='cpu'):
        if noise_schedule != "linear":
            raise NotImplementedError("only noise_schedule='linear' (what scripts/inference.py uses)")
        self.model = model
        self.device = device
        self.schedule = _AlphasCumprodSchedule(diffusion_steps)
        self._graphs: Dict[tuple, tuple] = {}
        owner = getattr(model, "__self__", model)              # the nn.Module behind a bound forward_with_dpmsolver
        self._params = list(owner.parameters()) if isinstance(owner, torch.nn.Module) else []

    # ---- host side: everything that does not depend on the latents
    def plan(self, S: int, eta) -> List[dict]:
        """Per denoiser evaluation i at time ts[i], ts = linspace(1, 1/N, S + 1): the model-input time and the scalars of
        pxa_sa_solver_step -- sigma, 1/alpha at ts[i]; the corrector of step i (has_corr, cA, c0, c1, cN; tau_c) and the
        predictor of step i + 1 (pA, p0, p1, pN; tau_p; order 1 at the first and last step, else 2; tau = 0 at the last)."""
        if S < 2:
            raise ValueError(f"S must be >= 2 (the predictor / corrector orders are 2), got {S}")
        sch = self.schedule
        ts = torch.linspace(sch.T, 1. / sch.total_N, S + 1)               # skip_type='time', skip_order=1
        tau = lambda t: eta if 0.2 <= t <= 0.8 else 0                     # float32 t against 0.2 / 0.8, as the reference
        plan = []
        for i in range(S):
            t = ts[i]
            st = dict(t_input=float((t - 1. / sch.total_N) * 1000.), sigma=float(sch.sigma(t)), inv_alpha=float(1. / sch.alpha(t)),
                      has_corr=i >= 1, tau_c=0, cA=0., c0=0., c1=0., cN=0.)
            if i >= 1:
                st["tau_c"] = tau(t)
                A, (c0, c1), N = _sa_update(sch, 2, st["tau_c"], [ts[j] for j in range(max(0, i - 2), i)], t, True)
                st.update(cA=float(A), c0=float(c0), c1=float(c1), cN=float(N))
            step = i + 1
            order = 1 if step in (1, S) else 2
            st["tau_p"] = 0 if step == S else tau(ts[step])
            A, g, N = _sa_update(sch, order, st["tau_p"], [ts[j] for j in range(max(0, i - 1), i + 1)], ts[step], False)
            st.update(pA=float(A), p0=float(g[0]), p1=float(g[1]) if order == 2 else 0., pN=float(N), order=order)
            plan.append(st)
        return plan

    # ---- device side
    def _draw(self, buf: torch.Tensor) -> None:
        """One of the loop's standard-normal draws (the reference's `torch.randn_like(x)`), into `buf`."""
        buf.normal_()

    def _run(self, x, x_pred, x0_prev, noise, plan, t_dev, cond, guided, cfg, model_kwargs, draw) -> torch.Tensor:
        draw(noise[0])                                   # the reference draws once before the first evaluation, unused
        for i, (st, t_in) in enumerate(zip(plan, t_dev)):
            out = self.model(torch.cat([x_pred, x_pred]) if guided else x_pred, t_in, cond, **model_kwargs)
            if out.dtype not in (torch.float32, torch.bfloat16):
                out = out.float()
            if not (out.stride(3) == 1 and out.stride(2) == out.shape[3] and out.stride(1) == out.shape[2] * out.shape[3]):
                out = out.contiguous()
            draw(noise[(i + 1) % 2])                     # the noise of step i + 1, drawn after evaluation i as in the reference
            lib.sa_solver_step(out, x, x_pred, x0_prev, noise[i % 2], noise[(i + 1) % 2], guided=guided, cfg_scale=cfg,
                               sigma=st["sigma"], inv_alpha=st["inv_alpha"], has_corr=st["has_corr"], cA=st["cA"],
                               c0=st["c0"], c1=st["c1"], cN=st["cN"], pA=st["pA"], p0=st["p0"], p1=st["p1"], pN=st["pN"])
        return x_pred

    @torch.no_grad()
    def sample(self, S, batch_size, shape, conditioning=None, callback=None, normals_sequence=None, img_callback=None,
               quantize_x0=False, eta=0., mask=None, x0=None, temperature=1., noise_dropout=0., score_corrector=None,
               corrector_kwargs=None, verbose=True, x_T=None, log_every_t=100, unconditional_guidance_scale=1.,
               unconditional_conditioning=None, model_kwargs={}, *, cuda_graph=False, **kwargs):
        """Returns (x, None), x the fp32 sample of shape x_T.shape.  Like the reference, the arguments between `callback`
        and `log_every_t` other than `eta`, `x_T` are accepted and ignored.  x_T None: drawn with
        `torch.randn((batch_size,) + shape, device=device)` first.  cuda_graph=True: capture the loop once per configuration
        and replay it (x_T is drawn outside the graph; each replay draws fresh noise from the generator)."""
        plan = self.plan(S, eta)
        C, H, W = shape
        if x_T is None:
            if torch.device(self.device).type != "cuda":
                raise RuntimeError("pixart_sigma_b200.sampler has no CPU path: construct SASolverSampler with a CUDA device")
            x_T = torch.randn((batch_size, C, H, W), device=self.device)
        if not x_T.is_cuda:
            raise RuntimeError("pixart_sigma_b200.sampler has no CPU path: x_T must be a CUDA tensor")
        if x_T.dim() != 4 or x_T.shape[1] != 4 or (x_T.shape[2] * x_T.shape[3]) % 4:
            raise ValueError("latents must be (n, 4, h, w) with h*w a multiple of 4")
        if x_T.dtype != torch.float32:
            raise ValueError("x_T must be float32 (the loop's noise draws take its dtype)")
        guided = not (unconditional_guidance_scale == 1. or unconditional_conditioning is None)
        cond = torch.cat([unconditional_conditioning, conditioning]) if guided else conditioning    # [uncond ; cond]
        rows = 2 * x_T.shape[0] if guided else x_T.shape[0]
        t_dev = [torch.full((rows,), st["t_input"], dtype=torch.float32, device=x_T.device) for st in plan]
        cfg = float(unconditional_guidance_scale) if guided else 1.0
        if cuda_graph:
            return self._sample_graphed(x_T, plan, t_dev, cond, guided, cfg, model_kwargs, S, eta), None
        x_pred = x_T.contiguous().clone()
        x, x0_prev = torch.empty_like(x_pred), torch.empty_like(x_pred)
        noise = [torch.empty_like(x_pred), torch.empty_like(x_pred)]
        return self._run(x, x_pred, x0_prev, noise, plan, t_dev, cond, guided, cfg, model_kwargs, self._draw), None

    def _sample_graphed(self, x_T, plan, t_dev, cond, guided, cfg, model_kwargs, S, eta):
        # the plan's scalars and t_input are baked into the captured kernel arguments and the model_kwargs tensors into the
        # captured forward (by address): all of them are part of the key.  x_T and the conditioning (a new tensor per call)
        # are copied into the graph's own input buffers.
        key = (tuple(x_T.shape), x_T.device.index, guided, cfg, tuple(cond.shape), cond.dtype,
               _captured_model_key(self.model, self._params, model_kwargs), S, eta,
               tuple(tuple(v for k, v in sorted(st.items())) for st in plan))
        if key not in self._graphs:
            bufs = [torch.empty_like(x_T) for _ in range(6)]               # z_in, x, x_pred, x0_prev, 2 x noise
            z_in, x, x_pred, x0_prev = bufs[:4]
            cond_in = cond.clone()
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):        # warm-up outside capture (lazy inits), zero noise: the generator is untouched
                x_pred.copy_(x_T)
                self._run(x, x_pred, x0_prev, bufs[4:], plan[:2], t_dev[:2], cond_in, guided, cfg, model_kwargs, torch.Tensor.zero_)
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                x_pred.copy_(z_in)
                self._run(x, x_pred, x0_prev, bufs[4:], plan, t_dev, cond_in, guided, cfg, model_kwargs, self._draw)
            self._graphs[key] = (graph, z_in, cond_in, x_pred, bufs, t_dev)
        graph, z_in, cond_in, x_pred = self._graphs[key][:4]
        z_in.copy_(x_T)
        cond_in.copy_(cond)
        graph.replay()
        return x_pred.clone()
