"""Measure the SA-Solver sampler (pixart_sigma_b200.sampler.SASolverSampler) on one GPU and print one JSON line.

Workload: the `--sampling_algo sa-solver` default of scripts/inference.py -- 25 steps, eta = 1, CFG 4.5 -- around
PixArt-Sigma-XL/2 at 1024 px (latent 128 x 128, 4096 tokens), 4 images (CFG batch 8), 300-token captions, seeded random
weights (the zero-initialised output layers un-zeroed as in bench.py).  Reports, as milliseconds per 25-step sample:
  * eager: the sampler without a graph;
  * graphed: `cuda_graph=True` (noise draws, 25 forwards and 25 step kernels replayed as one graph);
  * forwards: 25 replays of `graph.GraphedForward` alone, the denoiser floor of any 25-evaluation sampler;
  * overhead per step = (sample - forwards) / 25 for both.
Also the step kernel's time and achieved bandwidth from CUDA events around a graph of many back-to-back launches (its
working set, ~10 MB, stays in the 126 MB L2 between launches, as it does in the sampler), the library launches per
evaluation and the graphed-vs-eager agreement under the same seed.  GPU name and power limit are read in the same run.
    python tools/sa_sampler_bench.py [--reps 3] [--kernel-iters 500]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIDE, IMGS, L, PE, S, ETA, CFG = 128, 4, 300, 2.0, 25, 1, 4.5


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (q.stdout.strip().split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(), "unknown")
    return name, power


def timed_ms(fn, reps):
    """Mean device time of fn() over `reps` calls (events around the whole window, after a synchronise)."""
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=500)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tools/sa_sampler_bench.py measures on a GPU; none is visible")
    from pixart_sigma_b200 import PixArtMS_XL_2, lib
    from pixart_sigma_b200.graph import GraphedForward
    from pixart_sigma_b200.sampler import SASolverSampler
    dev = "cuda"
    name, power = gpu_info()
    torch.manual_seed(1234)
    with torch.device(dev):
        model = PixArtMS_XL_2(input_size=SIDE, pe_interpolation=PE, model_max_length=L)
        for blk in model.blocks:
            torch.nn.init.normal_(blk.cross_attn.proj.weight, std=0.02)
        torch.nn.init.normal_(model.final_layer.linear.weight, std=0.02)
    model = model.to(torch.bfloat16).eval()
    g = torch.Generator().manual_seed(99)
    y = torch.randn(2 * IMGS, 1, L, 4096, generator=g).to(torch.bfloat16).to(dev)
    lens = torch.randint(8, L + 1, (IMGS,), generator=g)
    mask = (torch.arange(L)[None] < lens[:, None]).long().to(dev)
    kw = dict(data_info=None, mask=mask)
    solver = SASolverSampler(model.forward_with_dpmsolver, device=dev)
    call = dict(S=S, batch_size=IMGS, shape=(4, SIDE, SIDE), conditioning=y[IMGS:], eta=ETA, unconditional_guidance_scale=CFG,
                unconditional_conditioning=y[:IMGS], model_kwargs=kw)

    with torch.no_grad():
        solver.sample(**call)                                                        # warm-up
        n0 = lib.launch_count()
        torch.manual_seed(7)
        eager_out, _ = solver.sample(**call)
        launches_per_eval = (lib.launch_count() - n0) / S
        torch.manual_seed(7)
        graphed_out, _ = solver.sample(**call, cuda_graph=True)                      # capture + replay
        agree_max = float((graphed_out - eager_out).abs().max())
        agree_rel = float((graphed_out - eager_out).norm() / eager_out.norm())
        ms_eager = timed_ms(lambda: solver.sample(**call), args.reps)
        ms_graph = timed_ms(lambda: solver.sample(**call, cuda_graph=True), args.reps)

        fwd = GraphedForward(model)
        x8 = torch.randn(2 * IMGS, 4, SIDE, SIDE, device=dev)
        ts = [torch.full((2 * IMGS,), st["t_input"], device=dev) for st in solver.plan(S, ETA)]
        for t in ts[:3]:
            fwd(x8, t, y, mask)
        ms_fwd = timed_ms(lambda: [fwd(x8, t, y, mask) for t in ts], args.reps)

        out = model.forward_with_dpmsolver(x8, ts[0], y, **kw)                      # the view the sampler hands the kernel
        st = solver.plan(S, ETA)[10]
        bufs = [torch.randn(IMGS, 4, SIDE, SIDE, device=dev) for _ in range(5)]
        step = lambda: lib.sa_solver_step(out, *bufs, guided=True, cfg_scale=CFG, **{k: st[k] for k in (
            "sigma", "inv_alpha", "has_corr", "cA", "c0", "c1", "cN", "pA", "p0", "p1", "pN")})
        for _ in range(10):
            step()
        # back-to-back launches from one graph: a host loop of ctypes calls would time the enqueue rate, not the kernel
        chain = torch.cuda.CUDAGraph()
        with torch.cuda.graph(chain):
            for _ in range(args.kernel_iters):
                step()
        chain.replay()
        us_step = timed_ms(chain.replay, 5) * 1e3 / args.kernel_iters
    elems = IMGS * 4 * SIDE * SIDE
    bytes_step = elems * (2 * out.element_size() + 5 * 4 + 3 * 4)   # eps_u, eps_c; x, x_pred, x0_prev, noise x2; 3 writes
    res = {
        "what": "SA-Solver 25-step eta=1 CFG-4.5 sample, PixArt-Sigma-XL/2 1024px, 4 images (CFG batch 8), seeded random weights",
        "gpu": name, "power_limit": power,
        "ms_per_sample": {"eager": ms_eager, "graphed": ms_graph, "forwards_only_25x_GraphedForward": ms_fwd},
        "overhead_ms_per_step": {"eager": (ms_eager - ms_fwd) / S, "graphed": (ms_graph - ms_fwd) / S},
        "step_kernel": {"us": us_step, "bytes": bytes_step, "GB_per_s": bytes_step / (us_step * 1e-6) / 1e9,
                        "model_out_dtype": str(out.dtype), "launches_timed": 5 * args.kernel_iters, "timing": "events around 5 replays of a graph of back-to-back launches",
                        "note": "working set ~%.0f MB, L2-resident between launches" % (bytes_step / 1e6)},
        "library_launches_per_evaluation": launches_per_eval,
        "graphed_vs_eager_same_seed": {"max_abs": agree_max, "rel": agree_rel},
        "reps": args.reps,
    }
    print(json.dumps(res))


if __name__ == "__main__":
    main()
