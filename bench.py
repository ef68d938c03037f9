#!/usr/bin/env python
"""bench.py -- denoise-steps/sec of the PixArt-Sigma-XL/2 denoiser hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3|c2|c4|c5|vae|t5] [--impl ours|reference] [--no-extras]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Headline (`value`, workload c3 = BASELINE configs[2]'s per-GPU slice): a *step* is one pass of the hot path over one batch --
one `PixArtMS.forward` of the CFG-batched latents of the images a GPU holds (4 images/GPU at 1024px -> forward batch 8,
4096 tokens/sample), i.e. one DPM-Solver model evaluation.  `value` = image-denoise-steps per second over all ranks (an
image-step = one forward at batch 2, reference diffusion/model/dpm_solver.py:328-331), inputs resident in HBM, CUDA-event
timed, max over ranks.  `e2e` is the same metric through the public API with pinned HOST inputs copied H2D and the eps result
copied D2H inside every timed step.  Weak scaling: per-GPU work is fixed, ranks are independent replicas (no collective in
the data path, SURVEY.md 8e).  The working set per step (1.2 GB of weights + >1 GB of activations) is far larger than the
126 MB L2, so no explicit L2 flush is needed between iterations.

Nothing but the forward runs inside the timed region of `value`: the per-kernel CUDA events behind `roofline` are taken in a
SEPARATE pass afterwards, and after the timed regions rank 0 checks what it timed -- `parity` = rel. error of one
PixArtMSBlock at the benchmarked geometry (and, at N = 1, of the whole 28-block forward of one image) against the oracle
evaluated on the host.

The same invocation also puts BASELINE configs[4] (training step: IDDPM loss fwd + bwd + DDP gradient all-reduce, key
`train`) and configs[3] (2K, KV-compress sr=2, key `c4`) under the same clock at the same N (skip with --no-extras), so that
the scaling harness sees the NCCL gradient all-reduce too.

`--workload vae` / `--workload t5` time the callers either side of the denoiser (SURVEY.md 8f.2 / 8f.4): the SDXL-VAE decode of one
1024 x 1024 image (`value` = the ResBlock / upsample convolution stack, `e2e` = the whole `AutoencoderKL.decode` from a pinned-host
latent to the image read back) and one T5-v1.1-XXL forward over 4 captions x 300 tokens, each with its kernel roofline and a bounded
CPU sample of the reference's own path (diffusers is absent: the oracle decoder; transformers' T5EncoderModel).  `c5 --no-fp32-attention`
leaves the `fp32_attention` flag of the reference's 1024px config off (it selects the hi + lo P form of the attention forward).

One JSON line is printed by rank 0.

`--dump-outputs DIR` writes, after the timed steps, what the timed path handed its caller in its LAST timed step as
`DIR/<name>.npy` (float32, rank 0): `eps` (the forward's noise prediction; `c4_eps` for the extra c4 line), `loss` and `grads`
(the training step's mean loss and the gradients of all parameters in `named_parameters` order, flattened; `train_` prefix for
the extra line), `stack_out` (vae) and `last_hidden_state` (t5).  An array of more than DUMP_MAX_ELEMS elements is replaced by
the same seeded sample of its flattened elements in every run.  Weights and inputs come from fixed seeds, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

C, L, HEADS, DEPTH = 1152, 300, 16, 28
CPU_THREADS = 32            # fixed: torch CPU GEMMs of this size stop scaling long before the box's core count
WORKLOADS = {
    # name: (description, latent side, images per GPU, pe_interpolation, kv-compress)
    "c2": ("c2: PixArt-Sigma-XL/2 512px, 4 images/GPU (forward batch 8, CFG pairs), 1024 tokens", 64, 4, 1.0, False),
    "c3": ("c3: PixArt-Sigma-XL/2 1024-MS, 4 images/GPU (forward batch 8, CFG pairs), 4096 tokens "
           "[BASELINE configs[2]: batch 32 sharded over 8 GPUs]", 128, 4, 2.0, False),
    "c4": ("c4: PixArt-Sigma-XL/2 2K-MS kv-compress sr=2 layers 14-27, 1 image/GPU (forward batch 2), 16384 tokens "
           "[BASELINE configs[3]]", 256, 1, 4.0, True),
    "c5": ("c5: PixArt-Sigma-XL/2 1024-MS training step: IDDPM loss fwd + bwd (per-block activation checkpointing) + "
           "bucketed gradient all-reduce, 4 images/GPU, 4096 tokens, fp32 master weights / bf16 kernels "
           "[BASELINE configs[4]]", 128, 4, 2.0, False),
}


def flops_per_forward(n_tok: int, batch: int, kv_compress: bool):
    """Algorithmic FLOPs of one forward (SURVEY.md 8d): per block 28NC^2 + 4LC^2 + 4N Nk C + 4NLC; returns
    (total, gemm part, attention part)."""
    gemm_blk = 28 * n_tok * C * C + 4 * L * C * C
    tot_gemm = tot_attn = 0
    for i in range(DEPTH):
        nk = n_tok // 4 if (kv_compress and i >= 14) else n_tok
        tot_gemm += gemm_blk
        tot_attn += 4 * n_tok * nk * C + 4 * n_tok * L * C
    emb = 2 * L * 4096 * C + 2 * L * C * C + 2 * n_tok * 16 * C + 2 * n_tok * C * 32 + (2 * 256 * C + 14 * C * C)
    return batch * (tot_gemm + tot_attn + emb), batch * (tot_gemm + 2 * L * 4096 * C + 2 * L * C * C), batch * tot_attn


DUMP_SEED, DUMP_MAX_ELEMS, DUMP_MAX_BYTES = 0, 1 << 23, 64 << 20


def dump_array(t: torch.Tensor) -> np.ndarray:
    """`t` as float32 on the host; above DUMP_MAX_ELEMS elements, the DUMP_SEED-seeded sample of its flattened elements."""
    t = t.detach()
    if t.numel() > DUMP_MAX_ELEMS:
        idx = torch.randint(0, t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(DUMP_SEED))
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu().numpy()


def write_outputs(out_dir: str, outputs: dict) -> None:
    assert outputs and sum(a.nbytes for a in outputs.values()) <= DUMP_MAX_BYTES, {k: a.nbytes for k, a in outputs.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name).read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for nm, v in zip(names, r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        # "under load" = samples drawing more than half the observed max power
        load = [s for s, pw in zip(sm, power) if power and pw > 0.5 * max(power)] or sm
        return {"sm_mhz": statistics.median(load) if load else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(rows), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------- distributed context
class Ctx:
    def __init__(self, gpus: int, dump: bool = False):
        import torch.distributed as dist
        self.dist = dist
        self.last_output, self.outputs = None, {}
        self.rank, self.world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world == 1 and gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.dumping = dump and self.rank == 0

    def keep(self, name: str, t: torch.Tensor) -> None:
        """Record `t` for --dump-outputs (rank 0 only)."""
        if self.dumping:
            self.outputs[name] = dump_array(t)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps: int) -> float:
        """EXACTLY `steps` calls between two CUDA events, barrier + synchronize on both sides, max over ranks (ms).
        What the last call returned is left in `last_output`."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            out = fn(i)
        e1.record()
        self.barrier()
        self.last_output = out
        ms = e0.elapsed_time(e1)
        if self.world > 1:
            tt = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(tt, op=self.dist.ReduceOp.MAX)
            ms = float(tt.item())
        return ms

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


# --------------------------------------------------------------------------------------------- CPU arm (oracle)
def _oracle_cfg(po, side, pe, kv, depth=DEPTH):
    layers = list(range(14, 28)) if kv else []
    return po.OracleConfig(depth=depth, input_size=side, pe_interpolation=pe, kv_sampling="conv" if kv else None,
                           kv_scale_factor=2 if kv else 1, kv_compress_layer=layers)


def cpu_reference_forward(side: int, pe: float, kv: bool, sd=None, inputs=None, reps: int = 1):
    """ONE REAL timed forward of the oracle port of the reference `PixArtMS.forward` (fp32, torch CPU, CPU_THREADS threads)
    at the workload's resolution: forward batch 2 = one image with CFG, all 28 blocks (SURVEY.md 8d).  With `sd` / `inputs`
    it runs on the benchmarked model's own (bf16-valued) weights and inputs so that its output doubles as the parity
    reference of the GPU forward.  Returns (image-steps/s, seconds per forward, output)."""
    from oracle import pixart_oracle as po            # bench.py may use the oracle ONLY in the CPU arms / parity check
    torch.set_num_threads(min(os.cpu_count() or 1, CPU_THREADS))
    cfg = _oracle_cfg(po, side, pe, kv)
    if sd is None:
        sd = po.synthetic_state_dict(cfg, seed=0)
    if inputs is None:
        x, t, y, mask = po.synthetic_inputs(cfg, 2, (side, side), lens=[300, 300])
    else:
        x, t, y, mask = inputs
    with torch.no_grad():
        po.forward(sd, _oracle_cfg(po, side, pe, kv, depth=0), x, t, y, mask=mask)      # warm-up: embedders, thread pool
        times, out = [], None
        for _ in range(reps):
            t0 = time.perf_counter()
            out = po.forward(sd, cfg, x, t, y, mask=mask)
            times.append(time.perf_counter() - t0)
    sec = statistics.median(times)
    return 1.0 / sec, sec, out


def cpu_reference_train_sample(side: int, pe: float):
    """Training counterpart (workload c5): the oracle port of the reference forward with autograd + the IDDPM loss +
    backward (fp32, CPU), ONE image, through a 1-block and a 3-block slice of the 28-block model; per-block time =
    (t3 - t1) / 2, fixed = t1 - per-block, full step = fixed + 28 x per-block (a full fwd + bwd of one image would take
    minutes).  Returns (images/s, seconds measured)."""
    from oracle import pixart_oracle as po
    from pixart_sigma_b200.training import IDDPMLoss
    torch.set_num_threads(min(os.cpu_count() or 1, CPU_THREADS))

    def run(depth):
        cfg = po.OracleConfig(depth=depth, input_size=side, pe_interpolation=pe)
        sd = {k: v.requires_grad_(v.is_floating_point()) for k, v in po.synthetic_state_dict(cfg, seed=0).items()}
        x, _, y, mask = po.synthetic_inputs(cfg, 1, (side, side), lens=[300])
        model = lambda xx, timestep, **kw: po.forward_grad(sd, cfg, xx, timestep.float(), kw["y"], mask=kw["mask"])
        t0 = time.perf_counter()
        terms = IDDPMLoss().training_losses(model, x * 0.5, torch.tensor([500]), dict(y=y, mask=mask, data_info=None),
                                            noise=torch.randn_like(x))
        terms["loss"].mean().backward()
        return time.perf_counter() - t0

    run(0)                                             # warm-up (embedders, thread pool)
    t1, t3 = run(1), run(3)
    per_block = max((t3 - t1) / 2.0, 1e-9)
    fixed = max(t1 - per_block, 0.0)
    return 1.0 / (fixed + DEPTH * per_block), t1 + t3


def cpu_reference_t5_sample(caps: int, L: int):
    """`--workload t5`: the reference's own CPU path is transformers' T5EncoderModel (diffusion/model/t5.py:12,107-110).  A full
    T5-v1.1-XXL forward on the host needs 19 GB of fp32 weights and minutes, so the bounded sample is a 1-block and a 3-block model of
    XXL width (d_model 4096, 64 heads, d_ff 10240; fp32, CPU_THREADS threads) on the same `caps` x L token ids: per-block time =
    (t3 - t1) / 2, full forward = fixed + 24 x per-block.  Returns (captions/s, seconds measured)."""
    import transformers
    torch.set_num_threads(min(os.cpu_count() or 1, CPU_THREADS))

    def run(layers):
        cfg = transformers.T5Config(vocab_size=512, d_model=4096, d_kv=64, d_ff=10240, num_layers=layers, num_heads=64,
                                    feed_forward_proj="gated-gelu", dropout_rate=0.0)
        m = transformers.T5EncoderModel(cfg).eval()
        ids = torch.randint(0, 512, (caps, L), generator=torch.Generator().manual_seed(1))
        with torch.no_grad():
            m(input_ids=ids[:, :8])                                  # warm-up: thread pool, lazy initialisation
            t0 = time.perf_counter()
            m(input_ids=ids, attention_mask=torch.ones_like(ids))
            return time.perf_counter() - t0

    t1, t3 = run(1), run(3)
    per_block = max((t3 - t1) / 2.0, 1e-9)
    fixed = max(t1 - per_block, 0.0)
    return caps / (fixed + 24 * per_block), t1 + t3


def cpu_reference_vae_sample():
    """`--workload vae`: diffusers is not installed, so the CPU arm is the oracle's restatement of the SDXL-VAE decoder
    (oracle/vae_oracle.py, fp32, CPU_THREADS threads) on a 32 x 32 latent -> 256 x 256 image: 1 / 16 of the pixels of the benchmarked
    1024 x 1024 decode (every layer is per-pixel work except the mid-block attention, 6 % of the FLOPs at 1024 px, which grows with the
    square); images/s = 1 / (16 x t).  Returns (images/s, seconds measured)."""
    from oracle import vae_oracle as vo             # bench.py may use the oracle ONLY in the CPU arms / parity check
    from pixart_sigma_b200.vae import AutoencoderKL
    torch.set_num_threads(min(os.cpu_count() or 1, CPU_THREADS))
    torch.manual_seed(0)
    sd = {k: v.float() for k, v in AutoencoderKL().state_dict().items() if k.startswith(("decoder.", "post_quant_conv."))}
    z = torch.randn(1, 4, 32, 32)
    with torch.no_grad():
        vo.decode(sd, z[:, :, :8, :8])                                # warm-up
        t0 = time.perf_counter()
        vo.decode(sd, z)
        dt = time.perf_counter() - t0
    return 1.0 / (16.0 * dt), dt


def run_reference_arm(args, wl):
    """`--impl reference`: the reference's own CPU path (its oracle port: the reference is pure Python and cannot travel),
    same workload string / metric / unit as our arm; every step is one REAL forward of one image (forward batch 2)."""
    desc, side, imgs, pe, kv = wl
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = min(os.cpu_count() or 1, CPU_THREADS)
    train = args.workload == "c5"
    timed = max(1, min(args.steps, 3))
    if train:
        vals = [cpu_reference_train_sample(side, pe) for _ in range(timed)]
        value, sec = statistics.median(v for v, _ in vals), sum(s for _, s in vals)
        sample = (f"oracle port of the reference training step (forward with autograd + IDDPM loss + backward, fp32 torch CPU, "
                  f"{threads} threads), {side * 8}px, one image: 1- and 3-block slices timed, full step = fixed + 28 x "
                  f"per-block; median of {timed}, {sec:.1f} s of CPU work")
    else:
        value, sec, _ = cpu_reference_forward(side, pe, kv, reps=timed)
        sample = (f"oracle port of the reference PixArtMS.forward (fp32, torch CPU, {threads} threads), {side * 8}px: {timed} "
                  f"REAL full forward(s) of one image with CFG (forward batch 2, 28 blocks), median {sec:.2f} s each")
    unit = "images/s" if train else "image-steps/s"
    line = {"impl": "reference", "metric": "train-images/sec" if train else "denoise-steps/sec", "value": value, "unit": unit,
            "n_gpus": args.gpus, "steps": timed, "warmup": 1, "steps_requested": args.steps, "ms_per_step": 1000.0 / value,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "note": "reference is pure Python; its CPU path timed via the oracle port (the "
                       "reference itself cannot travel to the GPU box); per-image throughput of one host, not scaled by n_gpus"},
            "cpu_baseline": {"value": value, "unit": unit, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


# --------------------------------------------------------------------------------------------- our arm: inference
def run_reference_arm_callers(args):
    """`--impl reference --workload t5|vae`: the CPU path of the callers.  t5: transformers' T5EncoderModel itself (the reference's
    dependency, `kind: reference`), bounded to a 1-block + 3-block sample of XXL width per step and extrapolated to 24 blocks; vae:
    diffusers is not installed, so the oracle's decoder (`kind: port`) on a 256 x 256 image scaled to 1024 x 1024.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    steps = max(1, min(args.steps, 3))
    vals, secs = [], []
    for _ in range(steps):
        v, dt = cpu_reference_t5_sample(4, 300) if args.workload == "t5" else cpu_reference_vae_sample()
        vals.append(v)
        secs.append(dt)
    v = statistics.median(vals)
    t5 = args.workload == "t5"
    unit = "captions/s" if t5 else "images/s"
    wl = ("t5: T5-v1.1-XXL encoder forward (24 layers, d_model 4096, 64 heads, d_ff 10240), 4 captions x 300 tokens per GPU, random-init weights"
          if t5 else "vae: SDXL-VAE decode of one 1024x1024 image per GPU (whole AutoencoderKL.decode), random weights")
    cpu = {"value": v, "unit": unit, "cores": min(os.cpu_count() or 1, CPU_THREADS), "kind": "reference" if t5 else "port",
           "sample": ("transformers T5EncoderModel, fp32 torch CPU, XXL width, 1-block + 3-block models on 4 x 300 tokens, extrapolated to 24 blocks"
                      if t5 else "oracle restatement of the SDXL-VAE decoder, fp32 torch CPU, 32 x 32 latent -> 256 x 256 image, scaled by 16")
                     + f" ({statistics.median(secs):.1f} s measured per step)"}
    _emit({"impl": "reference", "metric": "t5-xxl captions/sec" if t5 else "vae-decoder images/sec", "value": v, "unit": unit,
           "n_gpus": args.gpus, "steps": steps, "warmup": 0, "steps_requested": args.steps, "ms_per_step": (4.0 if t5 else 1.0) / v * 1000.0,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": wl}, "cpu_baseline": cpu,
           "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


class KernelTimer:
    """CUDA-event timing of every GEMM / attention launch on the launching stream (the separate roofline pass)."""

    def __init__(self, lib, names):
        self.lib, self.on = lib, False
        self.recs = {k: [] for k, _ in names}
        self._orig = {}
        for kind, fn_name in names:
            self._orig[fn_name] = getattr(lib, fn_name)
            setattr(lib, fn_name, self._make(kind, self._orig[fn_name]))

    def _make(self, kind, fn):
        def wrapped(*a, **k):
            if not self.on:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            self.recs[kind].append((e0, e1))
            return r
        return wrapped

    def restore(self):
        for name, fn in self._orig.items():
            setattr(self.lib, name, fn)

    def totals_ms(self):
        return {k: (sum(a.elapsed_time(b) for a, b in v), len(v)) for k, v in self.recs.items()}


def _block_parity(model, B, side, lens_cfg, dev):
    """One PixArtMSBlock of the benchmarked model at the benchmarked geometry (fused path, the kernels the timed region
    ran) against the oracle block on the host, on seeded inputs.  Returns the normwise rel. error of the block output."""
    from oracle import pixart_oracle as po
    from pixart_sigma_b200.model import _LnFusion, _ln_ctx, _LN_FUSE_MIN_ROWS
    blk = model.blocks[0]
    hw = (side // 2, side // 2)
    N = hw[0] * hw[1]
    sr = blk.attn.sr_ratio
    g = torch.Generator().manual_seed(2024)
    x = torch.randn(B, N, C, generator=g)
    t0 = torch.randn(B, 6 * C, generator=g) * 0.3
    lens = [int(v) for v in lens_cfg]
    ycat = torch.randn(sum(lens), C, generator=g).to(torch.bfloat16)
    sd = {"blocks.0." + k: v.detach().float().cpu() for k, v in blk.state_dict().items()}
    mod = (sd["blocks.0.scale_shift_table"][None] + t0.view(B, 6, C)).to(dev).contiguous()
    kv_len = torch.tensor(lens, dtype=torch.int32, device=dev)
    kv_off = torch.tensor([sum(lens[:i]) for i in range(B)], dtype=torch.int32, device=dev)
    ln = None
    if model.fuse_ln_modulate and N >= _LN_FUSE_MIN_ROWS:
        u, v, one_plus = _LnFusion([blk]).prepare(t0.view(B, 6, C).to(dev), mod[None], blk._ws)
        ln = _ln_ctx(u, v, one_plus, 0, torch.empty(B * N, 8, 2, device=dev))
    with torch.no_grad():
        got = blk.run_kernels(x.reshape(B * N, C).to(dev).contiguous(), ycat.to(dev), kv_len, kv_off, max(lens), mod, B, N, hw,
                              blk._ws, ln).view(B, N, C).cpu()
        torch.set_num_threads(min(os.cpu_count() or 1, 64))
        want = po.block_forward(sd, "blocks.0", x, ycat.float()[None], t0, lens, hw, HEADS, sr, blk.attn.sampling if sr > 1 else None)
    return po.rel_err(got, want), po.rel_err(got - x, want - x)


def measure_inference(args, ctx: Ctx, wl_name: str, headline: bool):
    from pixart_sigma_b200 import PixArtMS_XL_2, lib
    desc, side, imgs, pe, kv = WORKLOADS[wl_name]
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(1234 + rank)
    kvc = dict(sampling="conv", scale_factor=2, kv_compress_layer=list(range(14, 28))) if kv else None
    with torch.device(dev):
        model = PixArtMS_XL_2(input_size=side, pe_interpolation=pe, model_max_length=L, kv_compress_config=kvc)
        for blk in model.blocks:                      # un-zero the zero-initialised layers (SURVEY.md 8d weights)
            torch.nn.init.normal_(blk.cross_attn.proj.weight, std=0.02)
        torch.nn.init.normal_(model.final_layer.linear.weight, std=0.02)
    model = model.to(torch.bfloat16).eval()

    B = 2 * imgs                                       # CFG: [uncond, cond] per image
    n_tok = (side // 2) ** 2
    # DPM-Solver time grid of a 20-step run: (linspace(1, 1e-3, 21)[:-1] - 1e-3) * 1000 = 999.0, 949.05, ...
    tgrid = ((torch.linspace(1.0, 1e-3, 21)[:-1] - 1e-3) * 1000.0).tolist()
    g = torch.Generator().manual_seed(99 + rank)
    h_x = torch.randn(B, 4, side, side, generator=g).pin_memory()
    h_y = torch.randn(B, 1, L, 4096, generator=g).to(torch.bfloat16).pin_memory()
    lens = torch.randint(8, L + 1, (imgs,), generator=g)
    h_mask = (torch.arange(L)[None] < lens[:, None]).long().pin_memory()          # (imgs, L), repeated over CFG pairs
    h_t = torch.empty(B, dtype=torch.float32).pin_memory()
    h_out = torch.empty(B, 4, side, side, dtype=torch.bfloat16).pin_memory()
    d_x, d_y, d_mask = h_x.to(dev), h_y.to(dev), h_mask.to(dev)
    d_ts = [torch.full((B,), tv, device=dev) for tv in tgrid]

    graphed = None
    if args.cuda_graph:
        from pixart_sigma_b200.graph import GraphedForward
        graphed = GraphedForward(model)

    def step_resident(i):
        if graphed is not None:
            return graphed(d_x, d_ts[i % 20], d_y, d_mask)
        return model.forward_with_dpmsolver(d_x, d_ts[i % 20], d_y, None, mask=d_mask)

    def step_e2e(i):
        h_t.fill_(tgrid[i % 20])
        if graphed is not None:          # GraphedForward copies the (pinned host) arguments into its static device buffers
            eps = graphed(h_x, h_t, h_y, h_mask)
        else:
            x = h_x.to(dev, non_blocking=True); t = h_t.to(dev, non_blocking=True)
            y = h_y.to(dev, non_blocking=True); mk = h_mask.to(dev, non_blocking=True)
            eps = model.forward_with_dpmsolver(x, t, y, None, mask=mk)
        h_out.copy_(eps, non_blocking=True)
        return eps

    warm = max(args.warmup, 3)
    with torch.no_grad():
        n_pre = lib.launch_count()
        model.forward_with_dpmsolver(d_x, d_ts[0], d_y, None, mask=d_mask)          # eager: kernel launches of one forward
        launches_per_forward = lib.launch_count() - n_pre
        for i in range(warm):
            step_resident(i)
        step_e2e(0)
        sampler = ClockSampler(ctx.local) if rank == 0 else None
        if os.environ.get("PXA_PROFILER_RANGE") == "1":      # ncu --profile-from-start off: capture the timed steps only
            torch.cuda.profiler.start()
        ms = ctx.timed(step_resident, args.steps)                                   # <- `value`: nothing else in here
        if os.environ.get("PXA_PROFILER_RANGE") == "1":
            torch.cuda.profiler.stop()
        ctx.keep("eps" if headline else f"{wl_name}_eps", ctx.last_output)
        ms_e2e = ctx.timed(step_e2e, args.steps)
        clocks = sampler.stop() if sampler else None
        # ---- separate pass: per-kernel CUDA events for the roofline (2 steps; not part of value / e2e)
        timer = KernelTimer(lib, [("gemm", "gemm"), ("attn", "flash_attn")])
        timer.on = True
        roof_steps = 2
        ms_roof = ctx.timed(lambda i: model.forward_with_dpmsolver(d_x, d_ts[i % 20], d_y, None, mask=d_mask), roof_steps)
        timer.on = False
        timer.restore()
        loop = None
        if args.sampling_loop:
            # the caller of the path (SURVEY.md 8f.1): a full 20-step DPM-Solver++ CFG sampling run of `imgs` images
            from pixart_sigma_b200.sampler import DPMS
            cond, null = d_y[imgs:], d_y[:imgs]
            solver = DPMS(model.forward_with_dpmsolver, condition=cond, uncondition=null, cfg_scale=4.5,
                          model_kwargs=dict(data_info=None, mask=d_mask))
            z = d_x[:imgs].float()
            solver.sample(z, steps=20, cuda_graph=args.cuda_graph)                 # warm-up (and graph capture)
            ms_loop = ctx.timed(lambda i: solver.sample(z, steps=20, cuda_graph=args.cuda_graph), 1)
            loop = {"steps": 20, "images": imgs * world, "ms": ms_loop, "images_per_s": imgs * world / (ms_loop / 1000.0),
                    "denoise_steps_per_s": imgs * world * 20 / (ms_loop / 1000.0), "cuda_graph": bool(args.cuda_graph)}

    line = None
    if rank == 0:
        tot, f_gemm, f_attn = flops_per_forward(n_tok, B, kv)
        ms_step = ms / args.steps
        value = imgs * world * args.steps / (ms / 1000.0)
        e2e_v = imgs * world * args.steps / (ms_e2e / 1000.0)
        sus, burst, hbm, src = measured_peaks()
        tt = timer.totals_ms()
        gemm_ms, gemm_n = tt["gemm"]
        attn_ms, attn_n = tt["attn"]
        gemm_tf = f_gemm * roof_steps / (gemm_ms / 1000.0) / 1e12 if gemm_ms > 0 else None
        attn_tf = f_attn * roof_steps / (attn_ms / 1000.0) / 1e12 if attn_ms > 0 else None
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "latest_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic, traffic_src = tj.get("gemm_dram_bytes_per_launch"), tj.get("source")
        roof = {"bound": "tensor", "kernel": "pxa::gemm_bf16_kernel / gemm2_bf16_kernel (all GEMMs of the block; %.0f%% of the FLOPs)"
                % (100.0 * f_gemm / tot),
                "achieved": gemm_tf, "peak": sus, "unit": "TFLOP/s", "frac": (gemm_tf / sus) if gemm_tf else None,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src})", "traffic": traffic,
                "traffic_source": traffic_src,
                "timing": f"CUDA events around every launch in a separate {roof_steps}-step pass after the timed regions "
                          f"({ms_roof / roof_steps:.2f} ms/step with the events)",
                "launches_timed": gemm_n, "avg_launch_ms": gemm_ms / max(gemm_n, 1),
                "flops_per_launch_avg": f_gemm * roof_steps / max(gemm_n, 1),
                # shares of the TIMED step (graph replay), not of the eager events pass: on a slow host that pass is launch-bound
                # (its wall time grows, the kernels' durations do not)
                "step_share": gemm_ms / roof_steps / ms_step,
                "events_pass_host_bound": bool(ms_roof / roof_steps > 1.15 * ms_step),
                "attention": {"kernel": "pxa::flash_attn_d72_kernel", "achieved": attn_tf, "frac": (attn_tf / sus) if attn_tf else None,
                              "launches_timed": attn_n, "step_share": attn_ms / roof_steps / ms_step},
                "whole_step": {"achieved": tot / (ms_step / 1000.0) / 1e12, "frac": tot / (ms_step / 1000.0) / 1e12 / sus}}
        # ---- what was timed is checked: one block at the benchmarked geometry vs the oracle on the host
        parity = None
        if not args.no_parity:
            blk_lens = torch.cat([lens, lens]).tolist()
            e_blk, e_upd = _block_parity(model, B, side, blk_lens, dev)
            parity = {"block_rel_err": e_blk, "block_update_rel_err": e_upd,
                      "block": f"PixArtMSBlock 0 of the benchmarked model, B={B}, {n_tok} tokens, caption lengths {blk_lens}, vs "
                               "oracle.block_forward (fp32, host) on the same bf16-valued weights", "bar": 1e-3 if not kv else 1.5e-3}
        cpu = None
        if world == 1 and not args.no_cpu_baseline and headline:
            # one REAL forward of the reference port on this box's cores, on the benchmarked model's weights and the first
            # image's inputs; its output is also the parity reference of the whole GPU forward
            sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
            t_in = torch.full((2,), tgrid[0])
            xin, yin = torch.cat([h_x[:1], h_x[imgs:imgs + 1]]), torch.cat([h_y[:1], h_y[imgs:imgs + 1]]).float()
            v, sec, want = cpu_reference_forward(side, pe, kv, sd=sd, inputs=(xin.to(torch.bfloat16).float(), t_in, yin, h_mask[:1]))
            cpu = {"value": v, "unit": "image-steps/s", "cores": min(os.cpu_count() or 1, CPU_THREADS), "kind": "port",
                   "sample": f"oracle port of the reference PixArtMS.forward, fp32 torch CPU, {side * 8}px: ONE real full forward "
                             f"of one image with CFG (forward batch 2, 28 blocks) in {sec:.2f} s"}
            if parity is not None:
                from oracle import pixart_oracle as po
                model.output_dtype = torch.float32
                with torch.no_grad():
                    got = model(xin.to(dev), t_in.to(dev), yin.to(dev).to(torch.bfloat16), mask=h_mask[:1].to(dev)).cpu()
                model.output_dtype = None
                parity["forward_rel_err"] = po.rel_err(got, want)
                parity["forward"] = "whole 28-block forward of image 0 (forward batch 2) vs the oracle forward above; bar 1e-2"
        h2d = h_x.numel() * 4 + h_y.numel() * 2 + h_mask.numel() * 8 + h_t.numel() * 4
        launches = launches_per_forward * args.steps
        line = {"metric": "denoise-steps/sec", "value": value, "unit": "image-steps/s", "n_gpus": world,
                "steps": args.steps, "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": desc, "images_per_gpu": imgs, "forward_batch_per_gpu": B,
                           "tokens_per_sample": n_tok, "text_tokens": L, "parallelism": f"dp{world} (batch-sharded replicas)",
                           "l2": "inputs larger than L2 (weights 1.2 GB + activations per step); no flush needed",
                           "cuda_graph": bool(args.cuda_graph), "fused_ln_modulate": bool(model.fuse_ln_modulate),
                           "tflop_per_step_per_gpu": tot / 1e12},
                "e2e": {"value": e2e_v, "unit": "image-steps/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h_out.numel() * 2},
                "gpu_launches": launches, "clocks": clocks, "roofline": roof, "cpu_baseline": cpu, "parity": parity}
        if loop is not None:
            line["sampling_loop"] = loop
    del model
    torch.cuda.empty_cache()
    return line


# --------------------------------------------------------------------------------------------- our arm: training step
def measure_train(args, ctx: Ctx, mode: str, checkpoint: bool, cpu_baseline: bool):
    """BASELINE configs[4]: one training step = zero_grad + IDDPM loss forward + backward + gradient all-reduce.
    mode: 'eager' (bucket all-reduces overlap the backward), 'graph' (whole step replayed from one CUDA graph, all-reduce
    after the replay), 'graph-overlap' (collectives captured inside the graph)."""
    from pixart_sigma_b200 import build_model, lib
    from pixart_sigma_b200.parallel import GradBucketReducer
    from pixart_sigma_b200.training import GraphedTrainStep, IDDPMLoss, train_step

    desc, side, imgs, pe, _ = WORKLOADS["c5"]
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.manual_seed(1234)                                   # same initial weights on every rank (DDP replicas)
    with torch.device(dev):
        model = build_model(dict(type="PixArtMS_XL_2", input_size=side, pe_interpolation=pe, model_max_length=L),
                            use_grad_checkpoint=checkpoint, use_fp32_attention=not args.no_fp32_attention)
        # configs/pixart_sigma_config/PixArt_sigma_xl2_img1024_internalms.py:14,27: fp32_attention = True, grad_checkpointing = True;
        # the builder applies the flag together with checkpointing (builder.py:12-13), so --no-checkpoint runs have it off
        for blk in model.blocks:
            torch.nn.init.normal_(blk.cross_attn.proj.weight, std=0.02)
        torch.nn.init.normal_(model.final_layer.linear.weight, std=0.02)
    model = model.float().train()
    reducer = GradBucketReducer(model, compress="bf16" if args.bf16_reduce else None)
    loss_fn = IDDPMLoss()
    n_tok = (side // 2) ** 2
    g = torch.Generator().manual_seed(7 + rank)
    h_x = (torch.randn(imgs, 4, side, side, generator=g) * 0.5).pin_memory()
    h_y = torch.randn(imgs, 1, L, 4096, generator=g).to(torch.bfloat16).pin_memory()
    lens = torch.randint(8, L + 1, (imgs,), generator=g)
    h_mask = (torch.arange(L)[None] < lens[:, None]).to(torch.int16).view(imgs, 1, 1, L).pin_memory()   # train.py:192 layout
    h_t = torch.randint(0, 1000, (imgs,), generator=g).pin_memory()
    h_noise = torch.randn(imgs, 4, side, side, generator=g).pin_memory()
    d_x, d_y, d_mask, d_t, d_noise = (v.to(dev) for v in (h_x, h_y, h_mask, h_t, h_noise))

    n_pre = lib.launch_count()
    reducer.zero_grad()
    train_step(model, loss_fn, d_x, d_t, d_y, d_mask, noise=d_noise, reducer=reducer)     # eager: kernel launches of one step
    launches_eager = lib.launch_count() - n_pre
    graphed = None
    if mode != "eager":
        graphed = GraphedTrainStep(model, loss_fn, reducer, (d_x, d_t, d_y, d_mask, d_noise),
                                   capture_collectives=(mode == "graph-overlap"))

    def step_resident(i):
        if graphed is not None:
            return graphed(d_x, d_t, d_y, d_mask, d_noise)
        reducer.zero_grad()
        return train_step(model, loss_fn, d_x, d_t, d_y, d_mask, noise=d_noise, reducer=reducer)

    def step_e2e(i):
        x, y, mk, t, nz = (v.to(dev, non_blocking=True) for v in (h_x, h_y, h_mask, h_t, h_noise))
        if graphed is not None:
            return float(graphed(x, t, y, mk, nz))
        reducer.zero_grad()
        return float(train_step(model, loss_fn, x, t, y, mk, noise=nz, reducer=reducer))     # loss read back: D2H + sync

    warm = max(args.warmup, 3)
    for i in range(warm):
        loss0 = step_resident(i)
    step_e2e(0)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    t_host = time.perf_counter()
    ms = ctx.timed(step_resident, args.steps)
    host_total_ms = (time.perf_counter() - t_host) * 1000.0
    prefix = "" if args.workload == "c5" else "train_"
    ctx.keep(prefix + "loss", ctx.last_output)
    if ctx.dumping:
        ctx.keep(prefix + "grads", torch.cat([p.grad.reshape(-1) for p in model.parameters() if p.grad is not None]))
    ms_e2e = ctx.timed(step_e2e, args.steps)
    clocks = sampler.stop() if sampler else None
    # exposed part of the gradient all-reduce: the same step with the collective switched off (world > 1 only)
    exposed = None
    if world > 1:
        saved = reducer.world
        reducer.world = 1
        for i in range(2):
            step_resident(i)
        ms_nocomm = ctx.timed(step_resident, args.steps)
        reducer.world = saved
        exposed = {"ms_per_step_without_collective": ms_nocomm / args.steps,
                   "exposed_allreduce_ms_per_step": (ms - ms_nocomm) / args.steps}
    # separate pass: per-kernel CUDA events (eager mode only; not available inside a graph replay)
    tt = None
    if mode == "eager":
        timer = KernelTimer(lib, [("gemm", "gemm"), ("gemm_wgrad", "gemm_wgrad"), ("attn", "flash_attn"), ("attn_bwd", "flash_attn_bwd")])
        timer.on = True
        ms_roof = ctx.timed(step_resident, 2)
        timer.on = False
        timer.restore()
        tt = timer.totals_ms()
    peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30
    line = None
    if rank == 0:
        fwd, f_gemm, f_attn = flops_per_forward(n_tok, imgs, False)
        sus, burst, hbm, src = measured_peaks()
        ms_step = ms / args.steps
        model_tf = 3 * fwd / (ms_step / 1000.0) / 1e12
        roof = {"bound": "tensor", "whole_step": {"model_tflops": model_tf, "frac": model_tf / sus,
                                                   "note": "model FLOPs = 3 x forward (no recomputation counted)"},
                "peak": sus, "unit": "TFLOP/s", "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src})"}
        if tt is not None:
            recompute = 1 if checkpoint else 0
            gemm_ms = tt["gemm"][0] + tt["gemm_wgrad"][0]
            gemm_tf = (3 + recompute) * f_gemm * 2 / (gemm_ms / 1000.0) / 1e12 if gemm_ms > 0 else None
            afw_tf = f_attn * 2 / (tt["attn"][0] / 1000.0) / 1e12 if tt["attn"][0] > 0 else None      # recomputation reuses (o, lse)
            abw_tf = 3.5 * f_attn * 2 / (tt["attn_bwd"][0] / 1000.0) / 1e12 if tt["attn_bwd"][0] > 0 else None
            roof.update({"kernel": "pxa GEMM family (forward, recompute, dgrad and wgrad)", "achieved": gemm_tf,
                         "frac": gemm_tf / sus if gemm_tf else None, "step_share": gemm_ms / ms_roof,
                         "attention_fwd": {"achieved": afw_tf, "frac": afw_tf / sus if afw_tf else None, "step_share": tt["attn"][0] / ms_roof},
                         "attention_bwd": {"achieved": abw_tf, "frac": abw_tf / sus if abw_tf else None,
                                           "step_share": tt["attn_bwd"][0] / ms_roof,
                                           "note": "executed FLOPs (14 N Nk d incl. the dQ-pass recomputation); model FLOPs are 10 N Nk d"}})
        h2d = h_x.numel() * 4 + h_y.numel() * 2 + h_mask.numel() * 2 + h_t.numel() * 8 + h_noise.numel() * 4
        line = {"metric": "train-images/sec", "value": imgs * world * args.steps / (ms / 1000.0), "unit": "images/s",
                "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": desc, "images_per_gpu": imgs, "tokens_per_sample": n_tok, "text_tokens": L,
                           "parallelism": f"ddp{world} (bucketed NCCL all-reduce of {reducer.grad_bytes() / 1e9:.2f} GB "
                                          f"{'bf16' if args.bf16_reduce else 'fp32'} gradients per rank, {len(reducer.buckets)} buckets)",
                           "step_mode": mode, "grad_checkpointing": checkpoint,
                           "fp32_attention": bool(getattr(model.blocks[0].attn, "fp32_attention", False)),
                           "optimizer_step": "not included (fwd + bwd + all-reduce, as configs[4] states)",
                           "l2": "working set (2.4 GB fp32 weights + activations) larger than L2; no flush needed",
                           "tflop_model_per_step_per_gpu": 3 * fwd / 1e12, "peak_mem_gib": peak_mem, "loss": float(loss0),
                           "host_ms_per_step": host_total_ms / args.steps},
                "e2e": {"value": imgs * world * args.steps / (ms_e2e / 1000.0), "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
                "gpu_launches": launches_eager * args.steps, "clocks": clocks, "roofline": roof, "allreduce": exposed,
                "cpu_baseline": None}
        if cpu_baseline:
            v, dt = cpu_reference_train_sample(side, pe)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": min(os.cpu_count() or 1, CPU_THREADS), "kind": "port",
                                    "sample": f"oracle port of the reference training step (forward with autograd + IDDPM loss + "
                                              f"backward, fp32 torch CPU), {side * 8}px, one image: 1- and 3-block slices timed "
                                              f"({dt:.1f} s), full step = fixed + 28 x per-block"}
    reducer.remove()
    del model, reducer, graphed
    torch.cuda.empty_cache()
    return line


# --------------------------------------------------------------------------------------------- our arm: VAE decoder convs
VAE_STACK = (  # SDXL-VAE decoder (block_out 128/256/512/512, 2+1 ResBlocks per up block) for a 1024 x 1024 image: latent 128 x 128
    [("res", 512, 512)] * 2 +                                   # mid block (its single-head attention is not ours)
    [("res", 512, 512)] * 3 + [("up", 512, 512)] +              # up block 0  @128^2 -> 256^2
    [("res", 512, 512)] * 3 + [("up", 512, 512)] +              # up block 1  @256^2 -> 512^2
    [("res", 512, 256), ("res", 256, 256), ("res", 256, 256), ("up", 256, 256)] +   # up block 2  @512^2 -> 1024^2
    [("res", 256, 128), ("res", 128, 128), ("res", 128, 128)])  # up block 3  @1024^2


def measure_vae(args, ctx: Ctx):
    """SURVEY.md 8a row 19 / 8f.2: the convolution-bearing part of the SDXL-VAE decode of ONE 1024 x 1024 image per GPU --
    17 ResnetBlock2D (GroupNorm+SiLU -> conv3x3 twice, 1x1 shortcut where the width changes) and 3 upsample convolutions,
    random weights (diffusers' VAE weights are not available offline).  value = images/s over all ranks."""
    from pixart_sigma_b200 import lib
    from pixart_sigma_b200.vae import DecoderResBlock, UpsampleConv
    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    torch.manual_seed(5 + rank)
    mods, flops, side = [], 0.0, 128
    with torch.device(dev):
        for kind, cin, cout in VAE_STACK:
            if kind == "res":
                m = DecoderResBlock(cin, cout)
                flops += 2.0 * side * side * 9 * (cin * cout + cout * cout) + (2.0 * side * side * cin * cout if cin != cout else 0.0)
            else:
                m = UpsampleConv(cin)
                side *= 2
                flops += 2.0 * side * side * 9 * cin * cout
            mods.append(m.to(torch.bfloat16))
    x0 = torch.randn(1, 512, 128, 128, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)

    def step(i):
        h = x0
        for m in mods:
            h = m(h)
        return h

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    n0 = lib.launch_count()
    ms = ctx.timed(step, args.steps)
    launches = lib.launch_count() - n0
    ctx.keep("stack_out", ctx.last_output)
    clocks = sampler.stop() if sampler else None
    # e2e: the call scripts/inference.py:136 makes -- `vae.decode(latent / scaling_factor).sample` of the whole autoencoder (conv_in,
    # mid block incl. its 16384-token attention, the stack above, conv_norm_out, conv_out) with the latent copied from pinned host
    # memory and the image read back every step
    from pixart_sigma_b200.vae import AutoencoderKL
    with torch.device(dev):
        full = AutoencoderKL().to(torch.bfloat16)
    h_z = torch.randn(1, 4, 128, 128).pin_memory()
    h_img = torch.empty(1, 3, 1024, 1024, dtype=torch.bfloat16).pin_memory()

    def step_e2e(i):
        z = h_z.to(dev, non_blocking=True)
        img = full.decode(z / full.config.scaling_factor).sample
        h_img.copy_(img, non_blocking=True)
        return img

    for i in range(2):
        step_e2e(i)
    ms_e2e = ctx.timed(step_e2e, args.steps)
    del full
    timer = KernelTimer(lib, [("conv", "conv3x3_nhwc"), ("gn", "groupnorm_silu_nhwc"), ("gemm", "gemm")])
    timer.on = True
    ms_roof = ctx.timed(step, 2)
    timer.on = False
    timer.restore()
    line = None
    if rank == 0:
        sus, burst, hbm, src = measured_peaks()
        tt = timer.totals_ms()
        conv_ms, conv_n = tt["conv"]
        conv_flops = flops - sum(2.0 * (128 * 2 ** j) ** 2 * a * b for j, a, b in ((2, 512, 256), (3, 256, 128)))   # minus the two 1x1 shortcuts
        conv_tf = conv_flops * 2 / (conv_ms / 1000.0) / 1e12 if conv_ms > 0 else None
        # GroupNorm+SiLU: 2 reads + 1 write of every normalised NHWC image (bf16)
        gn_bytes, sd = 0.0, 128
        for kind, cin, cout in VAE_STACK:
            if kind == "res":
                gn_bytes += 6.0 * sd * sd * (cin + cout)
            else:
                sd *= 2
        gn_ms = tt["gn"][0]
        line = {"metric": "vae-decoder-conv-stack images/sec", "value": world * args.steps / (ms / 1000.0), "unit": "images/s",
                "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "vae: SDXL-VAE decoder ResBlock + upsample convolutions of one 1024x1024 image per GPU "
                                       "(17 ResnetBlock2D + 3 upsample convs, GroupNorm+SiLU kernels, random weights)",
                           "tflop_per_step_per_gpu": flops / 1e12, "l2": "activations up to 268 MB per layer: larger than L2"},
                "e2e": {"value": world * args.steps / (ms_e2e / 1000.0), "unit": "images/s", "ms_per_step": ms_e2e / args.steps,
                        "what": "AutoencoderKL.decode of one 128x128 latent -> 1024x1024 image (whole decoder incl. conv_in, mid-block "
                                "attention, conv_out), latent from pinned host memory, image read back",
                        "h2d_bytes_per_step": h_z.numel() * 4, "d2h_bytes_per_step": h_img.numel() * 2},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "pxa::gemm_bf16_kernel<kConv> (implicit-GEMM 3x3 convolution, 4-D TMA)",
                             "achieved": conv_tf, "peak": sus, "unit": "TFLOP/s", "frac": conv_tf / sus if conv_tf else None,
                             "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src})", "launches_timed": conv_n,
                             "step_share": conv_ms / ms_roof, "traffic": None,
                             "groupnorm_silu": {"bound": "hbm", "achieved_gbs": gn_bytes * 2 / (gn_ms / 1000.0) / 1e9 if gn_ms > 0 else None,
                                                "peak_gbs": hbm, "step_share": gn_ms / ms_roof},
                             "whole_step_tflops": flops / (ms / args.steps / 1000.0) / 1e12},
                "cpu_baseline": None}
        if world == 1 and not args.no_cpu_baseline:
            v, dt = cpu_reference_vae_sample()
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": min(os.cpu_count() or 1, CPU_THREADS), "kind": "port",
                                    "sample": f"oracle restatement of the SDXL-VAE decoder (diffusers is not installed), fp32 torch CPU, one 32 x 32 "
                                              f"latent -> 256 x 256 image in {dt:.1f} s, scaled by 16 to the 1024 x 1024 decode of `e2e`"}
    return line


# --------------------------------------------------------------------------------------------- our arm: T5 caption encoder
def measure_t5(args, ctx: Ctx):
    """SURVEY.md 8(f).4: one forward of the T5-v1.1-XXL caption encoder (24 layers, d_model 4096, 4.7 B random-init bf16 parameters:
    there is no checkpoint offline) over the captions of one c3 batch -- 4 captions x 300 tokens per GPU (diffusion/model/t5.py:107-110;
    the null caption is a stored embedding).  value = captions/s over all ranks; e2e = token ids / mask from pinned host memory and the
    (4, 300, 4096) embeddings read back."""
    from pixart_sigma_b200 import lib
    from pixart_sigma_b200.t5 import T5EncoderModel, T5_V1_1_XXL
    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    cfg, caps, L = T5_V1_1_XXL, 4, 300
    torch.manual_seed(11)
    with torch.device(dev):
        torch.set_default_dtype(torch.bfloat16)
        try:
            model = T5EncoderModel()
        finally:
            torch.set_default_dtype(torch.float32)
        for n_, p_ in model.named_parameters():
            if p_.dim() > 1:
                torch.nn.init.normal_(p_, std=(p_.shape[1] ** -0.5) if "shared" not in n_ else 1.0)
    g = torch.Generator().manual_seed(3 + rank)
    h_ids = torch.randint(0, cfg["vocab_size"], (caps, L), generator=g).pin_memory()
    lens = torch.randint(8, L + 1, (caps,), generator=g)
    h_mask = (torch.arange(L)[None] < lens[:, None]).long().pin_memory()
    d_ids, d_mask = h_ids.to(dev), h_mask.to(dev)
    h_out = torch.empty(caps, L, cfg["d_model"], dtype=torch.bfloat16).pin_memory()

    def step(i):
        return model(d_ids, d_mask)["last_hidden_state"]

    def step_e2e(i):
        out = model(h_ids.to(dev, non_blocking=True), h_mask.to(dev, non_blocking=True))["last_hidden_state"]
        h_out.copy_(out, non_blocking=True)
        return out

    warm = max(args.warmup, 3)
    for i in range(warm):
        step(i)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    n0 = lib.launch_count()
    ms = ctx.timed(step, args.steps)
    launches = lib.launch_count() - n0
    ctx.keep("last_hidden_state", ctx.last_output)
    clocks = sampler.stop() if sampler else None
    ms_e2e = ctx.timed(step_e2e, args.steps)
    timer = KernelTimer(lib, [("gemm", "gemm"), ("rms", "rmsnorm"), ("attn", "t5_attn")])
    timer.on = True
    ms_roof = ctx.timed(step, 2)
    timer.on = False
    timer.restore()
    line = None
    if rank == 0:
        sus, burst, hbm, src = measured_peaks()
        D, F_, inner, nl, M = cfg["d_model"], cfg["d_ff"], cfg["num_heads"] * cfg["d_kv"], cfg["num_layers"], caps * L
        gemm_flops = nl * 2.0 * M * (4 * D * inner + 3 * D * F_)
        attn_flops = nl * 4.0 * caps * cfg["num_heads"] * L * L * cfg["d_kv"]
        wbytes = nl * 2.0 * (4 * D * inner + 3 * D * F_)
        tt = timer.totals_ms()
        gemm_ms, gemm_n = tt["gemm"]
        gemm_tf = gemm_flops * 2 / (gemm_ms / 1000.0) / 1e12 if gemm_ms > 0 else None
        attn_ms = tt["attn"][0]
        line = {"metric": "t5-xxl captions/sec", "value": caps * world * args.steps / (ms / 1000.0), "unit": "captions/s",
                "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "t5: T5-v1.1-XXL encoder forward (24 layers, d_model 4096, 64 heads, d_ff 10240), 4 captions x 300 "
                                       "tokens per GPU, random-init weights",
                           "tflop_per_step_per_gpu": (gemm_flops + attn_flops) / 1e12, "weight_gb": wbytes / 1e9,
                           "l2": "9.4 GB of weights streamed per forward: larger than L2"},
                "e2e": {"value": caps * world * args.steps / (ms_e2e / 1000.0), "unit": "captions/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": h_ids.numel() * 8 + h_mask.numel() * 8, "d2h_bytes_per_step": h_out.numel() * 2},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "tensor", "kernel": "pxa::gemm_bf16_kernel (the 7 Linear layers of each T5 block; 99 % of the FLOPs)",
                             "achieved": gemm_tf, "peak": sus, "unit": "TFLOP/s", "frac": gemm_tf / sus if gemm_tf else None,
                             "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({src})", "launches_timed": gemm_n,
                             "step_share": gemm_ms / ms_roof, "traffic": None,
                             "weights_gbs": wbytes * 2 / (gemm_ms / 1000.0) / 1e9 if gemm_ms > 0 else None, "hbm_peak_gbs": hbm,
                             "rmsnorm_step_share": tt["rms"][0] / ms_roof,
                             "attention": {"impl": model.attn_impl, "kernel": "pxa::t5_attn_d64_kernel", "step_share": attn_ms / ms_roof,
                                           "achieved": attn_flops * 2 / (attn_ms / 1000.0) / 1e12 if attn_ms > 0 else None},
                             "whole_step_tflops": (gemm_flops + attn_flops) / (ms / args.steps / 1000.0) / 1e12},
                "cpu_baseline": None}
        if world == 1 and not args.no_cpu_baseline:
            v, dt = cpu_reference_t5_sample(caps, L)
            line["cpu_baseline"] = {"value": v, "unit": "captions/s", "cores": min(os.cpu_count() or 1, CPU_THREADS), "kind": "reference",
                                    "sample": f"transformers T5EncoderModel (the reference's dependency), fp32 torch CPU, XXL width, {caps} captions x "
                                              f"{L} tokens through a 1-block and a 3-block model ({dt:.1f} s measured), extrapolated to 24 blocks"}
    del model
    torch.cuda.empty_cache()
    return line


_JSON_FD = None


def _emit(line: dict) -> None:
    data = (json.dumps(line) + "\n").encode()
    os.write(_JSON_FD if _JSON_FD is not None else 1, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS) + ["vae", "t5"])
    ap.add_argument("--no-extras", action="store_true",
                    help="headline workload only (default: the c3 line also carries the c5 training step under `train` and "
                         "the c4 2K forward under `c4`, measured at the same N)")
    ap.add_argument("--train-mode", default="auto", choices=["auto", "eager", "graph", "graph-overlap"],
                    help="c5: how the step is issued; auto = one CUDA graph (all-reduce after the replay)")
    ap.add_argument("--no-checkpoint", action="store_true", help="c5: train without per-block activation checkpointing")
    ap.add_argument("--no-fp32-attention", action="store_true",
                    help="c5: leave fp32_attention off (the reference 1024px config sets it; it makes the self-attention forward "
                         "take P as bf16 hi + lo terms)")
    ap.add_argument("--bf16-reduce", action="store_true", help="c5: gradients travel as bf16 (1.22 GB instead of 2.44 GB)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-run oracle check of one block at the bench geometry")
    ap.add_argument("--sampling-loop", action="store_true",
                    help="also time one full 20-step DPM-Solver++ sampling run through pixart_sigma_b200.sampler "
                         "(extra key `sampling_loop`; not part of the timed region of `value` / `e2e`)")
    ap.add_argument("--no-cuda-graph", dest="cuda_graph", action="store_false",
                    help="issue the forward eagerly (default: `value` and `e2e` replay it as ONE CUDA graph through the "
                         "public pixart_sigma_b200.graph.GraphedForward: ~310 launches and their host work per step disappear)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy (float32)")
    ap.set_defaults(cuda_graph=True)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs records the GPU path: use it with --impl ours")
    # The contract is ONE JSON line on stdout.  Libraries write banners there too (NCCL prints its version line at the
    # first communicator init), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved fd.
    global _JSON_FD
    sys.stdout.flush()
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        if args.workload in ("vae", "t5"):
            run_reference_arm_callers(args)
            return
        run_reference_arm(args, WORKLOADS[args.workload])
        return
    from pixart_sigma_b200 import lib
    ctx = Ctx(args.gpus, dump=bool(args.dump_outputs))
    lib.load()
    train_mode = "graph" if args.train_mode == "auto" else args.train_mode
    if args.workload == "vae":
        line = measure_vae(args, ctx)
    elif args.workload == "t5":
        line = measure_t5(args, ctx)
    elif args.workload == "c5":
        line = measure_train(args, ctx, train_mode, not args.no_checkpoint, ctx.world == 1 and not args.no_cpu_baseline)
    else:
        line = measure_inference(args, ctx, args.workload, headline=True)
        if args.workload == "c3" and not args.no_extras:
            sub = argparse.Namespace(**vars(args))
            sub.no_cpu_baseline, sub.sampling_loop = True, False
            tr = measure_train(sub, ctx, train_mode, not args.no_checkpoint, False)
            sub.no_parity = True
            c4 = measure_inference(sub, ctx, "c4", headline=False)
            if ctx.rank == 0:
                keep = ("metric", "value", "unit", "ms_per_step", "config", "e2e", "roofline", "allreduce", "clocks", "gpu_launches",
                        "steps", "warmup")
                line["train"] = {k: tr[k] for k in keep if k in tr}
                line["c4"] = {k: c4[k] for k in keep if k in c4}
    if ctx.dumping:
        write_outputs(args.dump_outputs, ctx.outputs)
    if ctx.rank == 0:
        _emit(line)
    ctx.close()


if __name__ == "__main__":
    main()
