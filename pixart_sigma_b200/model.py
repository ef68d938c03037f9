"""Host-side mirror of the reference denoiser API on top of the sm_100a kernels.

`PixArtMS`, `PixArtMSBlock`, `PixArtMS_XL_2` keep the reference's constructor arguments, method signatures,
attribute names and `state_dict()` key layout (diffusion/model/nets/PixArtMS.py:49-293, PixArt_blocks.py:28-158,
205-221, 267-407; checkpoint keys tools/convert_pixart_to_diffusers.py:30-155), so `scripts/inference.py`,
the DPM-Solver / IDDPM wrappers and `load_state_dict` of a reference `.pth` work unchanged.  What differs is
*where the math runs*: every per-block op is a call into libpixart_sm100.so (see `lib.py`), the residual stream
is carried in fp32 between blocks, and nothing in `forward` synchronises with the host (cached positional table,
device-side key lengths instead of `.tolist()`).

There is deliberately no CPU / eager fallback: `forward` requires CUDA bf16 parameters and raises otherwise.
"""
from __future__ import annotations

import math
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import lib

__all__ = ["PixArtMS", "PixArtMSBlock", "PixArtMS_XL_2", "MODELS", "build_model", "install_into_reference"]


# ------------------------------------------------------------------------------------------------- registry
class _Registry:
    """Name -> constructor table with the two mmcv.Registry methods the reference uses (builder.py:5,11)."""

    def __init__(self, name: str):
        self.name, self.module_dict = name, {}

    def register_module(self, name: Optional[str] = None, force: bool = False, module=None):
        def _add(obj):
            self.module_dict[name or obj.__name__] = obj
            return obj
        return _add(module) if module is not None else _add

    def build(self, cfg, default_args: Optional[dict] = None):
        kw = dict(cfg)
        for k, v in (default_args or {}).items():
            kw.setdefault(k, v)
        ctor = kw.pop("type")
        return (self.module_dict[ctor] if isinstance(ctor, str) else ctor)(**kw)


MODELS = _Registry("models")


def set_grad_checkpoint(model, use_fp32_attention=False, gc_step=1):
    """diffusion/model/utils.py:28-35: mark EVERY submodule -- `grad_checkpointing` makes the blocks recompute their activations in
    the backward (autograd.py), `fp32_attention` selects the hi + lo P form of the self-attention forward (PixArt_blocks.py:145-147;
    DESIGN.md 4.2b), `grad_checkpointing_step` is stored for the callers that read it."""
    assert isinstance(model, nn.Module)

    def mark(m):
        m.grad_checkpointing, m.fp32_attention, m.grad_checkpointing_step = True, use_fp32_attention, gc_step
    model.apply(mark)


def build_model(cfg, use_grad_checkpoint=False, use_fp32_attention=False, gc_step=1, **kwargs):
    """Same call surface as diffusion/model/builder.py:8-14."""
    if isinstance(cfg, str):
        cfg = dict(type=cfg)
    model = MODELS.build(cfg, default_args=kwargs)
    if use_grad_checkpoint:
        set_grad_checkpoint(model, use_fp32_attention=use_fp32_attention, gc_step=gc_step)
    return model


# ------------------------------------------------------------------------------------------------- leaf modules
class _Mlp(nn.Module):
    """fc1 -> GELU(tanh) -> fc2; parameter names of timm 0.6.12 `Mlp` (PixArtMS.py:67)."""

    def __init__(self, in_features: int, hidden_features: int, out_features: Optional[int] = None):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features)
        self.act = nn.GELU(approximate="tanh")
        self.fc2 = nn.Linear(hidden_features, out_features or in_features)


class PatchEmbed(nn.Module):
    """Conv2d(k = s = patch) tokeniser (PixArtMS.py:22-46)."""

    def __init__(self, patch_size=2, in_chans=4, embed_dim=1152, bias=True):
        super().__init__()
        self.patch_size = (patch_size, patch_size) if isinstance(patch_size, int) else tuple(patch_size)
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=self.patch_size, stride=self.patch_size, bias=bias)


class TimestepEmbedder(nn.Module):
    """Sinusoid(256) -> Linear -> SiLU -> Linear (PixArt_blocks.py:267-309). Tiny; evaluated in fp32 by torch."""

    def __init__(self, hidden_size: int, frequency_embedding_size: int = 256):
        super().__init__()
        self.mlp = nn.Sequential(nn.Linear(frequency_embedding_size, hidden_size), nn.SiLU(),
                                 nn.Linear(hidden_size, hidden_size))
        self.frequency_embedding_size = frequency_embedding_size

    @staticmethod
    def timestep_embedding(t: torch.Tensor, dim: int, max_period: float = 10000.0) -> torch.Tensor:
        half = dim // 2
        freqs = torch.exp(-math.log(max_period) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
        ang = t[:, None].float() * freqs[None]
        return torch.cat([torch.cos(ang), torch.sin(ang)], dim=-1)

    def embed_fp32(self, t: torch.Tensor) -> torch.Tensor:
        f = self.timestep_embedding(t, self.frequency_embedding_size)
        h = F.silu(F.linear(f, self.mlp[0].weight.float(), self.mlp[0].bias.float()))
        return F.linear(h, self.mlp[2].weight.float(), self.mlp[2].bias.float())

    def forward(self, t):
        return self.embed_fp32(t).to(self.mlp[0].weight.dtype)


class SizeEmbedder(TimestepEmbedder):
    """One embedding per scalar of `s`, concatenated (PixArt_blocks.py:312-344)."""

    def __init__(self, hidden_size: int, frequency_embedding_size: int = 256):
        super().__init__(hidden_size, frequency_embedding_size)
        self.outdim = hidden_size

    def embed_fp32(self, s: torch.Tensor, bs: int) -> torch.Tensor:  # type: ignore[override]
        if s.ndim == 1:
            s = s[:, None]
        if s.shape[0] != bs:
            s = s.repeat(bs // s.shape[0], 1)
        b, d = s.shape
        e = TimestepEmbedder.embed_fp32(self, s.reshape(-1))
        return e.reshape(b, d * self.outdim)

    def forward(self, s, bs):
        return self.embed_fp32(s, bs).to(self.mlp[0].weight.dtype)


class CaptionEmbedder(nn.Module):
    """T5 feature projector 4096 -> C -> C with train-time caption dropout (PixArt_blocks.py:378-407)."""

    def __init__(self, in_channels, hidden_size, uncond_prob, token_num=120):
        super().__init__()
        self.y_proj = _Mlp(in_channels, hidden_size, hidden_size)
        self.register_buffer("y_embedding", torch.randn(token_num, in_channels) / in_channels ** 0.5)
        self.uncond_prob = uncond_prob

    def token_drop(self, caption, force_drop_ids=None):
        if force_drop_ids is None:
            drop = torch.rand(caption.shape[0], device=caption.device) < self.uncond_prob
        else:
            drop = force_drop_ids == 1
        return torch.where(drop[:, None, None, None], self.y_embedding.to(caption.dtype), caption)


class T2IFinalLayer(nn.Module):
    """LN -> modulate(table + t) -> Linear C -> p*p*out (PixArt_blocks.py:205-221)."""

    def __init__(self, hidden_size, patch_size, out_channels):
        super().__init__()
        self.norm_final = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.linear = nn.Linear(hidden_size, patch_size * patch_size * out_channels)
        self.scale_shift_table = nn.Parameter(torch.randn(2, hidden_size) / hidden_size ** 0.5)
        self.out_channels = out_channels


class MultiHeadCrossAttention(nn.Module):
    """Parameter holder for q_linear / kv_linear / proj (PixArt_blocks.py:28-58)."""

    def __init__(self, d_model, num_heads, attn_drop=0.0, proj_drop=0.0, **_):
        super().__init__()
        assert d_model % num_heads == 0, "d_model must be divisible by num_heads"
        self.d_model, self.num_heads, self.head_dim = d_model, num_heads, d_model // num_heads
        self.q_linear = nn.Linear(d_model, d_model)
        self.kv_linear = nn.Linear(d_model, d_model * 2)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(d_model, d_model)
        self.proj_drop = nn.Dropout(proj_drop)


class AttentionKVCompress(nn.Module):
    """Parameter holder for qkv / proj (+ sr conv, norm for KV compression; q_norm / k_norm) (PixArt_blocks.py:61-95)."""

    def __init__(self, dim, num_heads=8, qkv_bias=True, sampling="conv", sr_ratio=1, qk_norm=False, **_):
        super().__init__()
        assert dim % num_heads == 0
        self.num_heads, self.scale = num_heads, (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(0.0)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(0.0)
        self.sampling, self.sr_ratio = sampling, sr_ratio
        if sr_ratio > 1 and sampling == "conv":
            self.sr = nn.Conv2d(dim, dim, groups=dim, kernel_size=sr_ratio, stride=sr_ratio)
            self.sr.weight.data.fill_(1 / sr_ratio ** 2)
            self.sr.bias.data.zero_()
            self.norm = nn.LayerNorm(dim)
        if qk_norm:
            self.q_norm, self.k_norm = nn.LayerNorm(dim), nn.LayerNorm(dim)
        else:
            self.q_norm, self.k_norm = nn.Identity(), nn.Identity()


# ------------------------------------------------------------------------------------------------- workspace
class _Workspace:
    """Activation buffers reused by all 28 blocks of one forward (owned by the model, sized on first use)."""

    def __init__(self):
        self.key, self.buf = None, {}

    def get(self, name: str, shape: Tuple[int, ...], dtype: torch.dtype, device) -> torch.Tensor:
        t = self.buf.get(name)
        if t is None or t.shape != tuple(shape) or t.dtype != dtype or t.device != device:
            t = torch.empty(shape, dtype=dtype, device=device)
            self.buf[name] = t
        return t


_MLP_FUSED = os.environ.get("PXA_MLP_FUSED", "0") == "1"   # Mlp branch as one persistent kernel (mlp_sm100.cu)
_L2_CHAIN = os.environ.get("PXA_L2_CHAIN", "1") != "0"      # consumer kernels start on the rows their producer wrote last

_LN_FUSE_MIN_ROWS = 128      # a 128-row GEMM tile may span at most two samples (include/pixart_sm100.h)


def _ln_ctx(u: torch.Tensor, v: torch.Tensor, one_plus: torch.Tensor, i: int, stats: torch.Tensor) -> dict:
    """`ln` argument of PixArtMSBlock.run_kernels for block i of a chain (see _LnFusion.prepare)."""
    return {"stats": stats, "u": u[i], "v": v[i], "uv_stride": u.stride(1), "one_plus": one_plus[i], "prepare": i == 0,
            "next_one_plus": one_plus[i + 1] if i + 1 < one_plus.shape[0] else None}


class _KvBatch:
    """All `cross_attn.kv_linear` layers of the model as ONE GEMM per forward (PixArt_blocks.py:48: `self.kv_linear(cond)` with the
    same `cond` in every block).  28 GEMMs with M = B x text tokens (<= 2400 rows: 2 waves of half-empty tiles, 21 us each at c3)
    become one with N = depth x 2C (0.09 ms).  Owns the row-stacked weight / bias copies, rebuilt when a weight changes."""

    def __init__(self, blocks):
        self.blocks = list(blocks)
        self.key = None
        self.w = self.b = None

    def project(self, cond: torch.Tensor, ws: "_Workspace") -> torch.Tensor:
        mods = [blk.cross_attn.kv_linear for blk in self.blocks]
        key = tuple((m.weight._version, m.weight.data_ptr(), m.bias._version, m.bias.data_ptr()) for m in mods)
        if key != self.key:
            self.w = torch.cat([m.weight.detach() for m in mods], dim=0).contiguous()          # (depth * 2C, C)
            self.b = torch.cat([m.bias.detach() for m in mods], dim=0).contiguous()
            self.key = key
        out = ws.get("kv_all", (cond.shape[0], self.w.shape[0]), cond.dtype, cond.device)
        lib.gemm(cond, self.w, self.b, out)
        return out


# Opt-in (PXA_KV_BATCH=1): measured inside the noise at c3 (60.39 / 60.66 vs 60.61 ms -- the FLOPs are the same), and the stacked
# copy goes stale under in-place weight writes that bypass the version counter (`p.data.copy_()`: EMA / ZeRO-style updates).
_KV_BATCH = os.environ.get("PXA_KV_BATCH", "0") == "1"


class _LnFusion:
    """Per-forward conditioning of the FUSED LayerNorm-modulate (include/pixart_sm100.h, PXA_EPI_LN_BIAS).

    norm1 + t2i_modulate + attn.qkv (PixArtMS.py:75; PixArt_blocks.py:24-25,130) and norm2 + t2i_modulate + mlp.fc1
    (PixArtMS.py:77) are evaluated as  rstd_r * (A W^T - mu_r u_b) + v_b  in the GEMM epilogue, where A = bf16(x (1 + scale_b))
    and the row statistics come out of the residual epilogue that produced x.  This object owns what depends on the
    weights and the timestep only:
        u[i, b] = W_i (1 + scale_{i,b}),   v[i, b] = W_i shift_{i,b} + bias_i        for W_i in (qkv_i | fc1_i), fp32,
    with scale / shift = scale_shift_table_i + t0_b (adaLN-single: ONE t0 for all blocks).  The table part is static and
    computed once per weight version; the t0 part is ONE skinny GEMM per forward against the row-stacked weights of all
    blocks (a bf16 copy, 0.52 GB at depth 28), operands split into bf16 hi + lo parts so the result is fp32-accurate."""

    def __init__(self, blocks):
        self.blocks = list(blocks)
        self.key = None
        self.wstack = self.s_u = self.s_v = None

    def _weights(self):
        for blk in self.blocks:
            yield blk.attn.qkv
            yield blk.mlp.fc1

    @staticmethod
    def _split(t: torch.Tensor):
        hi = t.to(torch.bfloat16)
        return hi, (t - hi.float()).to(torch.bfloat16)

    def _skinny(self, rows: torch.Tensor, w: torch.Tensor, name: str, ws: "_Workspace") -> torch.Tensor:
        """fp32 (rows @ w.T) for a few fp32 rows: hi / lo bf16 split of the rows, one GEMM, reduce-add into a zeroed buffer."""
        hi, lo = self._split(rows)
        a = torch.cat([hi, lo], dim=0).contiguous()
        out = ws.get(name, (a.shape[0], w.shape[0]), torch.float32, w.device)
        out.zero_()
        lib.gemm(a, w, None, out, epilogue=lib.EPI_BIAS_RESIDUAL, residual=out)
        return out[: rows.shape[0]] + out[rows.shape[0]:]

    def _static(self, ws: "_Workspace"):
        mods = list(self._weights())
        key = tuple((m.weight._version, m.weight.data_ptr(), m.bias._version) for m in mods) + tuple(
            (b.scale_shift_table._version, b.scale_shift_table.data_ptr()) for b in self.blocks)
        if key == self.key:
            return
        w0 = mods[0].weight
        self.n1, self.n2 = mods[0].weight.shape[0], mods[1].weight.shape[0]
        self.ntot = self.n1 + self.n2
        self.wstack = torch.cat([m.weight.detach() for m in mods], dim=0).contiguous()          # (depth * ntot, C) bf16
        s_u, s_v = [], []
        for blk in self.blocks:
            tab = blk.scale_shift_table.detach().float()                                          # (6, C)
            for lin, i_shift, i_scale in ((blk.attn.qkv, 0, 1), (blk.mlp.fc1, 3, 4)):
                r = self._skinny(torch.stack([1.0 + tab[i_scale], tab[i_shift]]), lin.weight.detach(), "ln_static", ws)
                s_u.append(r[0].clone())
                s_v.append(r[1] + lin.bias.detach().float())
        depth = len(self.blocks)
        self.s_u = torch.cat(s_u).view(depth, self.ntot)
        self.s_v = torch.cat(s_v).view(depth, self.ntot)
        self.key = key

    def prepare(self, t0: torch.Tensor, mod_all: torch.Tensor, ws: "_Workspace"):
        """t0 (B, 6, C) fp32 (the t_block output), mod_all (depth, B, 6, C) = tables + t0.
        Returns u, v (depth, B, ntot) fp32 and one_plus (depth, B, 2, C) = 1 + (scale_msa | scale_mlp)."""
        self._static(ws)
        depth, B = mod_all.shape[0], mod_all.shape[1]
        # kind-major rows: shift_msa, scale_msa, shift_mlp, scale_mlp (plain slices: list indexing would copy an index tensor
        # from the host, which a CUDA-graph capture forbids)
        rows = torch.stack([t0[:, 0], t0[:, 1], t0[:, 3], t0[:, 4]]).reshape(4 * B, -1)
        g = self._skinny(rows, self.wstack, "ln_dyn", ws).view(4, B, depth, self.ntot)
        n1 = self.n1
        u = torch.cat([g[1, :, :, :n1], g[3, :, :, n1:]], dim=-1).permute(1, 0, 2) + self.s_u[:, None]
        v = torch.cat([g[0, :, :, :n1], g[2, :, :, n1:]], dim=-1).permute(1, 0, 2) + self.s_v[:, None]
        one_plus = 1.0 + torch.stack([mod_all[:, :, 1], mod_all[:, :, 4]], dim=2)
        return u.contiguous(), v.contiguous(), one_plus


def _drop_path_gates(mod: torch.Tensor, rate: float) -> torch.Tensor:
    """Stochastic depth (timm DropPath around the attention and MLP branches, PixArtMS.py:75,77): per sample, a branch is
    dropped with probability `rate` and the survivors are scaled by 1 / (1 - rate).  Both branches enter the residual stream
    through their gates, so DropPath is a per-sample factor on gate_msa (index 2) and gate_mlp (index 5) of `mod` (B, 6, C);
    the cross-attention branch has no DropPath in the reference (:76)."""
    keep = 1.0 - rate
    B = mod.shape[0]
    m = (torch.rand(B, 2, device=mod.device) < keep).to(mod.dtype) / keep
    scale = torch.ones(B, 6, 1, dtype=mod.dtype, device=mod.device)
    scale[:, 2, 0], scale[:, 5, 0] = m[:, 0], m[:, 1]
    return mod * scale


def _wants_grad(module: nn.Module, *inputs) -> bool:
    """True when autograd will record this call: grad mode on and a parameter or an input requires grad."""
    if not torch.is_grad_enabled():
        return False
    return any(p.requires_grad for p in module.parameters()) or any(
        isinstance(t, torch.Tensor) and t.requires_grad for t in inputs)


def _require_kernel_ready(p: torch.Tensor, what: str) -> None:
    if not p.is_cuda:
        raise RuntimeError(f"{what}: parameters are on {p.device}; pixart_sigma_b200 has no CPU path "
                           "(move the model to a B200 with .cuda())")
    if p.dtype != torch.bfloat16:
        raise RuntimeError(f"{what}: parameters are {p.dtype}; the sm_100a kernels take bf16 weights "
                           "(use model.to(torch.bfloat16))")


# ------------------------------------------------------------------------------------------------- block
class PixArtMSBlock(nn.Module):
    """adaLN-single DiT block: modulated self-attention, T5 cross-attention, modulated MLP (PixArtMS.py:49-79)."""

    def __init__(self, hidden_size, num_heads, mlp_ratio=4.0, drop_path=0.0, input_size=None, sampling=None,
                 sr_ratio=1, qk_norm=False, **block_kwargs):
        super().__init__()
        self.hidden_size = hidden_size
        self.norm1 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.attn = AttentionKVCompress(hidden_size, num_heads=num_heads, qkv_bias=True, sampling=sampling,
                                        sr_ratio=sr_ratio, qk_norm=qk_norm, **block_kwargs)
        self.cross_attn = MultiHeadCrossAttention(hidden_size, num_heads, **block_kwargs)
        self.norm2 = nn.LayerNorm(hidden_size, elementwise_affine=False, eps=1e-6)
        self.mlp = _Mlp(hidden_size, int(hidden_size * mlp_ratio))
        self.drop_path_rate = float(drop_path)
        self.drop_path = nn.Identity()
        self.scale_shift_table = nn.Parameter(torch.randn(6, hidden_size) / hidden_size ** 0.5)
        self._ws = _Workspace()
        self.__dict__["_ln_fusion"] = None        # built lazily by a stand-alone forward (not a submodule / state)

    # -- the fused path ---------------------------------------------------------------------------------------
    def run_kernels(self, x32: torch.Tensor, cond: torch.Tensor, kv_len: Optional[torch.Tensor],
                    kv_off: Optional[torch.Tensor], max_keys: int, mod: torch.Tensor, B: int, N: int,
                    HW: Tuple[int, int], ws: _Workspace, ln: Optional[dict] = None,
                    kv_pre: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One block on the kernels, in place on the fp32 residual stream.

        x32  (B*N, C) fp32 residual stream (updated in place and returned)
        cond (rows, C) bf16 embedded caption tokens; sample b's keys are rows kv_off[b] .. +kv_len[b]
             (kv_off None -> b*max_keys, kv_len None -> max_keys)
        mod  (B, 6, C) fp32 = scale_shift_table + t0  (shift_msa, scale_msa, gate_msa, shift_mlp, scale_mlp, gate_mlp)
        kv_pre  None, or this block's cross-attention keys / values (rows, 2C) bf16 (a strided view is fine) already projected by
             `_KvBatch` -- the caption tokens are the same for every block, so PixArtMS.forward runs all kv_linear layers as ONE GEMM.
        ln   None: norm + modulate as a stand-alone pass (pxa_ln_modulate) before the QKV / fc1 GEMMs.
             dict (from `_ln_ctx`): the FUSED form -- LayerNorm + t2i_modulate evaluated inside the QKV / fc1 GEMM epilogues
             from the scaled bf16 copy of x and the row statistics that the preceding residual epilogue left behind.
        """
        C, H = self.hidden_size, self.attn.num_heads
        M, dev = B * N, x32.device
        a, ca, mlp = self.attn, self.cross_attn, self.mlp
        _require_kernel_ready(a.qkv.weight, "PixArtMSBlock")
        bf = torch.bfloat16
        xn = ws.get("xn", (M, C), bf, dev)
        qkv = ws.get("qkv", (M, 3 * C), bf, dev)
        ao = ws.get("attn_o", (M, C), bf, dev)
        xb = ws.get("x_bf16", (M, C), bf, dev)
        ms = mod.stride(0)
        fused = ln is not None
        if fused:
            stats, u, v, one_plus, uvs = ln["stats"], ln["u"], ln["v"], ln["one_plus"], ln["uv_stride"]
            n1 = a.qkv.out_features
            lnkw = dict(ln_stats=stats, ln_uv_batch_stride=uvs, ln_dim=C, ln_eps=self.norm1.eps)

        # (1) x += gate_msa * proj(attn(LN(x) * (1 + scale_msa) + shift_msa))                     PixArtMS.py:75
        if fused:
            if ln["prepare"]:                       # first link of the chain: nobody has produced A / statistics for this x yet
                lib.ln_prepare(x32, one_plus[:, 0], xn, stats, mod_batch_stride=one_plus.stride(0), rows_per_batch=N)
            lib.gemm(xn, a.qkv.weight, None, qkv, epilogue=lib.EPI_LN_BIAS, rows_per_batch=N, ln_u=u[:, :n1], ln_v=v[:, :n1], **lnkw)
        else:
            lib.ln_modulate(x32, mod[:, 0], mod[:, 1], xn, mod_batch_stride=ms, rows_per_batch=N)
            lib.gemm(xn, a.qkv.weight, a.qkv.bias, qkv)
        if not isinstance(a.q_norm, nn.Identity):                                            # PixArt_blocks.py:133-134
            lib.layernorm_affine_(qkv[:, :C], a.q_norm.weight, a.q_norm.bias, eps=a.q_norm.eps)
            lib.layernorm_affine_(qkv[:, C:2 * C], a.k_norm.weight, a.k_norm.bias, eps=a.k_norm.eps)
        q3 = qkv.view(M, 3, H, C // H)
        k_src, v_src, k_str, n_keys = q3[:, 1], q3[:, 2], (3 * C, C // H), N
        if a.sr_ratio > 1:                                                                   # PixArt_blocks.py:137-139
            k_src, v_src, n_keys = self._compress_kv(qkv, B, N, HW, ws)
            k_str = (C, C // H)
        # L2 chaining (126 MB): each kernel starts on the rows its producer wrote last -- the QKV GEMM runs front to back, the
        # attention back to front (so attn.proj, front to back again, finds the first samples' outputs still cached)
        lib.flash_attn(q3[:, 0], k_src, v_src, ao, B=B, H=H, Nq=N, Nk=n_keys, kv_rows=B * n_keys,
                       q_strides=(3 * C, C // H), k_strides=k_str, v_strides=k_str, scale=a.scale, reverse_batch=_L2_CHAIN,
                       fp32_p=bool(getattr(a, "fp32_attention", False)))
        lib.gemm(ao, a.proj.weight, a.proj.bias, x32, epilogue=lib.EPI_BIAS_RESIDUAL, residual=x32, gate=mod[:, 2],
                 gate_batch_stride=ms, rows_per_batch=N, out_aux=xb)

        # (2) x += proj(cross_attn(x, cond))            (no norm, no gate)                       PixArtMS.py:76
        qx = ws.get("q_cross", (M, C), bf, dev)
        lib.gemm(xb, ca.q_linear.weight, ca.q_linear.bias, qx)
        if kv_pre is None:
            kv = ws.get("kv_cross", (cond.shape[0], 2 * C), bf, dev)
            lib.gemm(cond, ca.kv_linear.weight, ca.kv_linear.bias, kv)
        else:
            kv = kv_pre
        kv4 = kv.view(-1, 2, H, C // H)
        lib.flash_attn(qx, kv4[:, 0], kv4[:, 1], ao, B=B, H=H, Nq=N, Nk=max_keys, kv_rows=cond.shape[0],
                       kv_len=kv_len, kv_off=kv_off, q_strides=(C, C // H), k_strides=(kv.stride(0), C // H),
                       v_strides=(kv.stride(0), C // H), scale=(C // H) ** -0.5)
        if fused:       # the epilogue that produces x also leaves A = bf16(x (1 + scale_mlp)) and the row statistics of x
            lib.gemm(ao, ca.proj.weight, ca.proj.bias, x32, epilogue=lib.EPI_BIAS_RESIDUAL, residual=x32, rows_per_batch=N,
                     out_aux=xn, aux_scale=one_plus[:, 1], aux_scale_batch_stride=one_plus.stride(0), row_stats_out=stats)
        else:
            lib.gemm(ao, ca.proj.weight, ca.proj.bias, x32, epilogue=lib.EPI_BIAS_RESIDUAL, residual=x32)

        # (3) x += gate_mlp * fc2(gelu_tanh(fc1(LN(x) * (1 + scale_mlp) + shift_mlp)))           PixArtMS.py:77
        if self._mlp_one_kernel(N, M) and not fused:
            # the whole Mlp branch as ONE persistent GEMM -> GELU -> GEMM kernel, hidden activations resident in L2 (mlp_sm100.cu)
            lib.ln_modulate(x32, mod[:, 3], mod[:, 4], xn, mod_batch_stride=ms, rows_per_batch=N, reverse_rows=_L2_CHAIN)
            hws = ws.get("mlp_ring", (lib.MLP_RING * lib.MLP_GROUP * 256 * mlp.fc1.out_features,), bf, dev)
            fws = ws.get("mlp_flags", (3 * ((M + 255) // 256) + 8,), torch.int32, dev)
            lib.mlp_fused(xn, mlp.fc1.weight, mlp.fc1.bias, mlp.fc2.weight, mlp.fc2.bias, x32, gate=mod[:, 5], gate_batch_stride=ms,
                          rows_per_batch=N, hidden_ws=hws, flags_ws=fws)
            return x32
        hid = ws.get("mlp_hidden", (M, mlp.fc1.out_features), bf, dev)
        if fused:
            lib.gemm(xn, mlp.fc1.weight, None, hid, epilogue=lib.EPI_LN_BIAS_GELU, rows_per_batch=N, ln_u=u[:, n1:], ln_v=v[:, n1:],
                     **lnkw)
        else:
            # back to front: the rows of x the (front-to-back) cross-attention projection wrote last are still in L2
            lib.ln_modulate(x32, mod[:, 3], mod[:, 4], xn, mod_batch_stride=ms, rows_per_batch=N, reverse_rows=_L2_CHAIN)
            lib.gemm(xn, mlp.fc1.weight, mlp.fc1.bias, hid, epilogue=lib.EPI_BIAS_GELU)
        nxt = ln.get("next_one_plus") if fused else None
        if nxt is not None:                         # ... and here A / statistics for the NEXT block's norm1
            lib.gemm(hid, mlp.fc2.weight, mlp.fc2.bias, x32, epilogue=lib.EPI_BIAS_RESIDUAL, residual=x32, gate=mod[:, 5],
                     gate_batch_stride=ms, rows_per_batch=N, out_aux=xn, aux_scale=nxt[:, 0], aux_scale_batch_stride=nxt.stride(0),
                     row_stats_out=stats)
        else:       # back to front: the hidden rows fc1 wrote last (302 MB in all at c3) are the ones still in L2
            lib.gemm(hid, mlp.fc2.weight, mlp.fc2.bias, x32, epilogue=lib.EPI_BIAS_RESIDUAL, residual=x32, gate=mod[:, 5],
                     gate_batch_stride=ms, rows_per_batch=N, reverse_tiles=_L2_CHAIN)
        return x32

    def _mlp_one_kernel(self, N: int, M: int) -> bool:
        """Use pxa_mlp_fused_bf16 for the Mlp branch?  (PXA_MLP_FUSED=1; shapes the kernel is built for)"""
        return (_MLP_FUSED and N >= 128 and self.mlp.fc1.out_features % 256 == 0 and self.mlp.fc2.out_features % 192 == 0)

    def _compress_kv(self, qkv, B, N, HW, ws):
        """K / V token compression (PixArt_blocks.py:97-121). 'conv' sr=2 runs the fused conv+LN kernel; the
        parameter-free samplings are strided views materialised by torch (pure data movement)."""
        a, C = self.attn, self.hidden_size
        Hh, Ww = HW
        sr, dev = a.sr_ratio, qkv.device
        k_in, v_in = qkv[:, C:2 * C], qkv[:, 2 * C:]
        if a.sampling == "conv":
            if sr != 2:
                raise NotImplementedError("conv KV compression kernel is specialised for scale_factor 2")
            n_out = (Hh // 2) * (Ww // 2)
            kc = ws.get("k_comp", (B, n_out, C), torch.bfloat16, dev)
            vc = ws.get("v_comp", (B, n_out, C), torch.bfloat16, dev)
            lib.kv_compress(k_in, v_in, kc, vc, a.sr.weight, a.sr.bias, a.norm.weight, a.norm.bias, B=B, H=Hh, W=Ww,
                            ld_in=qkv.stride(0), eps=a.norm.eps)
            return kc.view(-1, C), vc.view(-1, C), n_out
        if a.sampling == "uniform_every":
            pick = lambda t: t.reshape(B, N, C)[:, ::sr].contiguous()
        elif a.sampling in ("uniform", "ave"):     # the reference's 'ave' is nearest-neighbour = the same strided pick
            pick = lambda t: t.reshape(B, Hh, Ww, C)[:, ::sr, ::sr].contiguous()
        else:
            raise ValueError(a.sampling)
        kc, vc = pick(k_in), pick(v_in)
        n_out = kc.numel() // (B * C)
        return kc.view(-1, C), vc.view(-1, C), n_out

    # -- reference call signature -------------------------------------------------------------------------------
    def forward(self, x, y, t, mask=None, HW=None, **kwargs):
        """x (B,N,C), y (1, sum(y_lens), C) packed caption tokens, t (B, 6C), mask = list y_lens (PixArtMS.py:71,206)."""
        B, N, C = x.shape
        if HW is None:
            HW = (int(N ** 0.5),) * 2
        cond = y.reshape(-1, C).to(torch.bfloat16).contiguous()
        if mask is None:
            lens = [cond.shape[0] // B] * B
        else:
            lens = [int(v) for v in mask]
        kv_len = torch.tensor(lens, dtype=torch.int32, device=x.device)
        kv_off = torch.tensor([sum(lens[:i]) for i in range(B)], dtype=torch.int32, device=x.device)
        mod = (self.scale_shift_table.float()[None] + t.reshape(B, 6, C).float()).contiguous()
        if self.training and self.drop_path_rate > 0:
            mod = _drop_path_gates(mod, self.drop_path_rate)
        x32 = x.reshape(B * N, C).float().contiguous()
        if _wants_grad(self, x, y, t):                                     # training: differentiable kernel ops
            from .autograd import block_train
            out = block_train(self, x32, cond, kv_len, kv_off, max(max(lens), 1), mod, B, N, tuple(HW),
                              bool(getattr(self, "grad_checkpointing", False)))
        else:
            _require_kernel_ready(self.attn.qkv.weight, "PixArtMSBlock")
            ln = None
            if N >= _LN_FUSE_MIN_ROWS and os.environ.get("PXA_FUSE_LN", "0") == "1":
                if self._ln_fusion is None:
                    self.__dict__["_ln_fusion"] = _LnFusion([self])
                u, v, one_plus = self._ln_fusion.prepare(t.reshape(B, 6, C).float(), mod[None], self._ws)
                ln = _ln_ctx(u, v, one_plus, 0, self._ws.get("ln_stats", (B * N, lib.LN_STAT_PARTS, 2), torch.float32, x.device))
            out = self.run_kernels(x32, cond, kv_len, kv_off, max(max(lens), 1), mod, B, N, tuple(HW), self._ws, ln)
        return out.view(B, N, C).to(x.dtype)


# ------------------------------------------------------------------------------------------------- model
_POS_CACHE: Dict[tuple, torch.Tensor] = {}


def _pos_embed_fp32(C: int, h: int, w: int, pe_interpolation: float, base_size: int, device) -> torch.Tensor:
    """(h*w, C) fp32 2-D sin/cos table, float64 math as the reference (PixArt.py:258-307), cached per geometry so the
    per-forward host computation + H2D copy of PixArtMS.py:177-182 happens once."""
    key = (C, h, w, float(pe_interpolation), int(base_size), str(device))
    tab = _POS_CACHE.get(key)
    if tab is None:
        pos_h = np.arange(h, dtype=np.float32) / (h / base_size) / pe_interpolation
        pos_w = np.arange(w, dtype=np.float32) / (w / base_size) / pe_interpolation
        omega = 1.0 / 10000 ** (np.arange(C // 4, dtype=np.float64) / (C // 4))
        aw = np.tile(pos_w[None, :], (h, 1)).reshape(-1)[:, None] * omega[None]     # w varies fastest
        ah = np.repeat(pos_h, w)[:, None] * omega[None]
        full = np.concatenate([np.sin(aw), np.cos(aw), np.sin(ah), np.cos(ah)], axis=1)
        tab = torch.from_numpy(full).to(torch.float32).to(device)
        _POS_CACHE[key] = tab
    return tab


@MODELS.register_module()
class PixArtMS(nn.Module):
    """Multi-scale PixArt-Sigma DiT (PixArtMS.py:85-285) running on the sm_100a kernels."""

    def __init__(self, input_size=32, patch_size=2, in_channels=4, hidden_size=1152, depth=28, num_heads=16,
                 mlp_ratio=4.0, class_dropout_prob=0.1, learn_sigma=True, pred_sigma=True, drop_path: float = 0.0,
                 caption_channels=4096, pe_interpolation=1.0, config=None, model_max_length=120,
                 micro_condition=False, qk_norm=False, kv_compress_config=None, **kwargs):
        super().__init__()
        self.pred_sigma = pred_sigma
        self.in_channels = in_channels
        self.out_channels = in_channels * 2 if pred_sigma else in_channels
        self.patch_size, self.num_heads, self.depth = patch_size, num_heads, depth
        self.pe_interpolation = pe_interpolation
        self.base_size = input_size // patch_size
        self.h = self.w = 0
        self.hidden_size = hidden_size
        # zero buffer kept only for checkpoint-key compatibility; the table is recomputed per geometry
        self.register_buffer("pos_embed", torch.zeros(1, self.base_size ** 2, hidden_size))
        self.x_embedder = PatchEmbed(patch_size, in_channels, hidden_size, bias=True)
        self.t_embedder = TimestepEmbedder(hidden_size)
        self.t_block = nn.Sequential(nn.SiLU(), nn.Linear(hidden_size, 6 * hidden_size, bias=True))
        self.y_embedder = CaptionEmbedder(caption_channels, hidden_size, class_dropout_prob, token_num=model_max_length)
        self.micro_conditioning = micro_condition
        if micro_condition:
            self.csize_embedder = SizeEmbedder(hidden_size // 3)
            self.ar_embedder = SizeEmbedder(hidden_size // 3)
        self.kv_compress_config = kv_compress_config or {"sampling": None, "scale_factor": 1, "kv_compress_layer": []}
        kvc = self.kv_compress_config
        rates = [float(v) for v in torch.linspace(0, drop_path, depth)]
        grid = (input_size // patch_size,) * 2
        self.blocks = nn.ModuleList([
            PixArtMSBlock(hidden_size, num_heads, mlp_ratio=mlp_ratio, drop_path=rates[i], input_size=grid,
                          sampling=kvc["sampling"],
                          sr_ratio=int(kvc["scale_factor"]) if i in kvc["kv_compress_layer"] else 1, qk_norm=qk_norm)
            for i in range(depth)])
        self.final_layer = T2IFinalLayer(hidden_size, patch_size, self.out_channels)
        self.output_dtype: Optional[torch.dtype] = None    # None -> model dtype (reference behaviour)
        # The reference casts `timestep` to the model dtype before the sinusoid (PixArtMS.py:174), which at bf16 turns
        # the DPM-Solver time 749.25 into 748 and moves the output by up to 5e-2 (SURVEY.md H6).  Default: keep the
        # timestep in fp32 like the fp32 reference does; set True to reproduce the bf16 cast bit for bit.
        self.round_timestep_to_dtype = False
        # True: LayerNorm + t2i_modulate inside the QKV / fc1 GEMM epilogues, no stand-alone norm pass (the north_star's
        # fusion; parity-tested at every geometry).  Default False = pxa_ln_modulate: measured on B200 in round 2 (DESIGN.md
        # 4.3) the fused chain is 0.3 ms / step SLOWER at c3 -- the read-modify-write residual epilogues that must produce
        # the scaled copy + row statistics (+23 / +41 us per block) and the extra epilogue work of the consuming GEMMs
        # (+13 / +39 us) cost more than the two 48 us passes they remove.  PXA_FUSE_LN=1 turns it on.
        self.fuse_ln_modulate = os.environ.get("PXA_FUSE_LN", "0") == "1"
        self.__dict__["_ln_fusion"] = None
        self.__dict__["_kv_batch"] = None
        self._ws = _Workspace()
        self.initialize()

    @property
    def dtype(self) -> torch.dtype:
        return next(self.parameters()).dtype

    # ---------------------------------------------------------------------------------------------------------
    def _condition(self, y: torch.Tensor, mask: Optional[torch.Tensor], B: int):
        """Caption embedding + key bookkeeping, all on device (replaces PixArtMS.py:194-204).

        Returns (cond (B*L, C) bf16, kv_len int32 (B,) or None, max_keys).  With a mask, each sample's selected
        tokens are moved to the front of its L-row slot (stable order), which is what masked_select packing feeds the
        block-diagonal attention -- softmax over a key *set* -- without the dynamic shape or the .tolist() sync."""
        ye, C = self.y_embedder, self.hidden_size
        L = y.shape[2]
        if self.training and ye.uncond_prob > 0:
            y = ye.token_drop(y)
        rows = y.reshape(B * L, -1).to(torch.bfloat16).contiguous()
        hid = self._ws.get("y_hidden", (B * L, C), torch.bfloat16, y.device)
        cond = self._ws.get("y_cond", (B * L, C), torch.bfloat16, y.device)
        lib.gemm(rows, ye.y_proj.fc1.weight, ye.y_proj.fc1.bias, hid, epilogue=lib.EPI_BIAS_GELU)
        lib.gemm(hid, ye.y_proj.fc2.weight, ye.y_proj.fc2.bias, cond)
        if mask is None:
            return cond, None, L
        if mask.shape[0] != B:
            mask = mask.repeat(B // mask.shape[0], *([1] * (mask.dim() - 1)))
        valid = mask.reshape(B, L) != 0
        order = torch.argsort((~valid).to(torch.uint8), dim=1, stable=True)              # selected tokens first
        cond = torch.gather(cond.view(B, L, C), 1, order[..., None].expand(B, L, C)).reshape(B * L, C)
        return cond, valid.sum(dim=1).to(torch.int32), L

    def forward(self, x, timestep, y, mask=None, data_info=None, **kwargs):
        """x (B, 4, H, W) latents, timestep (B,), y (B, 1, L, 4096) T5 features, mask (n, L) | (B,1,1,L) | None
        -> (B, 8, H, W)   (PixArtMS.py:165-211)."""
        w0 = self.blocks[0].attn.qkv.weight
        if _wants_grad(self, x, y):
            # the kernels fix their own precisions (bf16 operands, fp32 accumulation / statistics / residual stream); an
            # ambient autocast (accelerate's mixed precision, train.py:369) must not down-cast the fp32 torch glue around them
            with torch.autocast(device_type="cuda", enabled=False):
                return self._forward_train(x, timestep, y, mask=mask, data_info=data_info)
        if w0.is_cuda and w0.dtype == torch.float16:
            # scripts/inference.py:161 loads the checkpoint as fp16 (`weight_dtype = torch.float16`).  The sm_100a kernels
            # take bf16 operands, so the parameters are cast ONCE, in place; inputs / outputs keep the caller's fp16.
            import warnings
            warnings.warn("pixart_sigma_b200: fp16 parameters cast to bf16 for the sm_100a kernels (outputs stay fp16)")
            if self.output_dtype is None:
                self.output_dtype = torch.float16
            self.to(torch.bfloat16)
            w0 = self.blocks[0].attn.qkv.weight
        _require_kernel_ready(w0, "PixArtMS.forward")
        dt, dev, C, p = self.dtype, w0.device, self.hidden_size, self.patch_size
        B = x.shape[0]
        x = x.to(device=dev, dtype=dt)
        timestep = timestep.to(device=dev, dtype=dt if self.round_timestep_to_dtype else torch.float32)
        y = y.to(device=dev)
        if mask is not None:
            mask = mask.to(device=dev)
        self.h, self.w = x.shape[-2] // p, x.shape[-1] // p
        N = self.h * self.w

        pe = self.x_embedder.proj
        tok = F.conv2d(x.float(), pe.weight.float(), pe.bias.float(), stride=p).flatten(2).transpose(1, 2)
        x32 = (tok + _pos_embed_fp32(C, self.h, self.w, self.pe_interpolation, self.base_size, dev)[None])
        x32 = x32.reshape(B * N, C).contiguous()                                               # fp32 residual stream

        t = self.t_embedder.embed_fp32(timestep)                                               # (B, C) fp32
        if self.micro_conditioning:
            csize = self.csize_embedder.embed_fp32(data_info["img_hw"].to(dev, dt), B)
            ar = self.ar_embedder.embed_fp32(data_info["aspect_ratio"].to(dev, dt), B)
            t = t + torch.cat([csize, ar], dim=1)
        t0 = F.linear(F.silu(t), self.t_block[1].weight.float(), self.t_block[1].bias.float())  # (B, 6C) fp32
        tables = torch.stack([blk.scale_shift_table for blk in self.blocks]).float()           # (depth, 6, C)
        mod_all = (tables[:, None] + t0.view(1, B, 6, C)).contiguous()                          # (depth, B, 6, C)
        if self.training and any(blk.drop_path_rate > 0 for blk in self.blocks):
            mod_all = torch.stack([_drop_path_gates(mod_all[i], blk.drop_path_rate) if blk.drop_path_rate > 0 else mod_all[i]
                                   for i, blk in enumerate(self.blocks)])

        cond, kv_len, max_keys = self._condition(y, mask, B)
        fused = self.fuse_ln_modulate and N >= _LN_FUSE_MIN_ROWS and len(self.blocks) > 0
        if fused:
            if self._ln_fusion is None:
                self.__dict__["_ln_fusion"] = _LnFusion(self.blocks)
            u, v, one_plus = self._ln_fusion.prepare(t0.view(B, 6, C), mod_all, self._ws)
            stats = self._ws.get("ln_stats", (B * N, lib.LN_STAT_PARTS, 2), torch.float32, dev)
        kv_all = None
        if _KV_BATCH and len(self.blocks) > 1:
            if self._kv_batch is None:
                self.__dict__["_kv_batch"] = _KvBatch(self.blocks)
            kv_all = self._kv_batch.project(cond, self._ws)
        for i, blk in enumerate(self.blocks):
            blk.run_kernels(x32, cond, kv_len, None, max_keys, mod_all[i], B, N, (self.h, self.w), self._ws,
                            _ln_ctx(u, v, one_plus, i, stats) if fused else None,
                            None if kv_all is None else kv_all[:, i * 2 * C:(i + 1) * 2 * C])

        fl = self.final_layer                                                                  # uses t, not t0 (:208)
        fmod = (fl.scale_shift_table.float()[None] + t[:, None]).contiguous()                  # (B, 2, C): shift, scale
        xn = self._ws.get("xn", (B * N, C), torch.bfloat16, dev)
        lib.ln_modulate(x32, fmod[:, 0], fmod[:, 1], xn, mod_batch_stride=fmod.stride(0), rows_per_batch=N)
        out = F.linear(xn.float(), fl.linear.weight.float(), fl.linear.bias.float()).view(B, N, -1)
        return self.unpatchify(out).to(self.output_dtype or dt)

    def _forward_train(self, x, timestep, y, mask=None, data_info=None):
        """The same forward recorded for autograd (train_scripts/train.py:189-197): every block op is a
        `torch.autograd.Function` over the sm_100a kernels (autograd.py), blocks marked by `set_grad_checkpoint`
        (diffusion/model/utils.py:28-45) are activation-checkpointed like PixArtMS.py:206.  Parameters may be fp32
        (mixed precision: the kernels read cached bf16 shadows) or bf16."""
        from torch.utils.checkpoint import checkpoint
        from . import autograd as ag
        w0 = self.blocks[0].attn.qkv.weight
        if not w0.is_cuda:
            raise RuntimeError(f"PixArtMS: parameters are on {w0.device}; pixart_sigma_b200 has no CPU path")
        dt, dev, C, p = self.dtype, w0.device, self.hidden_size, self.patch_size
        B = x.shape[0]
        x = x.to(device=dev)
        timestep = timestep.to(device=dev, dtype=dt if self.round_timestep_to_dtype else torch.float32)
        y = y.to(device=dev)
        self.h, self.w = x.shape[-2] // p, x.shape[-1] // p
        N = self.h * self.w
        pe = self.x_embedder.proj
        tok = F.conv2d(x.float(), pe.weight.float(), pe.bias.float(), stride=p).flatten(2).transpose(1, 2)
        x32 = (tok + _pos_embed_fp32(C, self.h, self.w, self.pe_interpolation, self.base_size, dev)[None])
        x32 = x32.reshape(B * N, C).contiguous()
        t = self.t_embedder.embed_fp32(timestep)
        if self.micro_conditioning:
            csize = self.csize_embedder.embed_fp32(data_info["img_hw"].to(dev, dt), B)
            ar = self.ar_embedder.embed_fp32(data_info["aspect_ratio"].to(dev, dt), B)
            t = t + torch.cat([csize, ar], dim=1)
        t0 = F.linear(F.silu(t), self.t_block[1].weight.float(), self.t_block[1].bias.float())
        t0 = t0.view(B, 6, C)

        ye = self.y_embedder                                                # caption projector (PixArt_blocks.py:400-407)
        L = y.shape[2]
        if self.training and ye.uncond_prob > 0:
            y = ye.token_drop(y)
        rows = y.reshape(B * L, -1).to(torch.bfloat16)
        cond = ag.linear(ag.GeluFn.apply(ag.linear(rows, ye.y_proj.fc1)), ye.y_proj.fc2)
        kv_len = None
        if mask is not None:
            mask = mask.to(device=dev)
            if mask.shape[0] != B:
                mask = mask.repeat(B // mask.shape[0], *([1] * (mask.dim() - 1)))
            valid = mask.reshape(B, L) != 0
            order = torch.argsort((~valid).to(torch.uint8), dim=1, stable=True)
            cond = torch.gather(cond.view(B, L, C), 1, order[..., None].expand(B, L, C)).reshape(B * L, C)
            kv_len = valid.sum(dim=1).to(torch.int32)

        for blk in self.blocks:
            mod = blk.scale_shift_table.float()[None] + t0
            if self.training and blk.drop_path_rate > 0:        # drawn here, outside the (recomputed) checkpointed function
                mod = _drop_path_gates(mod, blk.drop_path_rate)
            # one autograd node per block (autograd.BlockFn, activation checkpointing built in) where it applies
            x32 = ag.block_train(blk, x32, cond, kv_len, None, L, mod, B, N, (self.h, self.w),
                                 bool(getattr(blk, "grad_checkpointing", False)))

        fl = self.final_layer
        fmod = (fl.scale_shift_table.float()[None] + t[:, None]).contiguous()
        xn = ag.LnModulateFn.apply(x32, fmod, 0, 1, N)
        out = F.linear(xn.float(), fl.linear.weight.float(), fl.linear.bias.float()).view(B, N, -1)
        return self.unpatchify(out).to(self.output_dtype or dt)

    def forward_with_dpmsolver(self, x, timestep, y, data_info, **kwargs):
        """DPM-Solver wants eps only: first half of the channels (PixArtMS.py:213-219)."""
        return self.forward(x, timestep, y, data_info=data_info, **kwargs).chunk(2, dim=1)[0]

    def forward_with_cfg(self, x, timestep, y, cfg_scale, data_info, mask=None, **kwargs):
        """Classifier-free guidance over a [cond | uncond] batch; like the reference, only the first THREE channels
        are mixed (PixArtMS.py:221-234)."""
        half = x[: len(x) // 2]
        out = self.forward(torch.cat([half, half], dim=0), timestep, y, mask, data_info=data_info, **kwargs)
        eps, rest = out[:, :3], out[:, 3:]
        cond_eps, uncond_eps = torch.split(eps, len(eps) // 2, dim=0)
        mixed = uncond_eps + cfg_scale * (cond_eps - uncond_eps)
        return torch.cat([torch.cat([mixed, mixed], dim=0), rest], dim=1)

    def unpatchify(self, x):
        """(B, h*w, p*p*c) -> (B, c, h*p, w*p) (PixArtMS.py:236-248)."""
        c, p = self.out_channels, self.x_embedder.patch_size[0]
        assert self.h * self.w == x.shape[1]
        x = x.reshape(x.shape[0], self.h, self.w, p, p, c)
        return x.permute(0, 5, 1, 3, 2, 4).reshape(x.shape[0], c, self.h * p, self.w * p)

    def initialize(self):
        """Same initial distribution as PixArtMS.initialize (PixArtMS.py:250-285)."""
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight)
                if m.bias is not None:
                    nn.init.zeros_(m.bias)
        w = self.x_embedder.proj.weight.data
        nn.init.xavier_uniform_(w.view(w.shape[0], -1))
        small = [self.t_embedder.mlp[0], self.t_embedder.mlp[2], self.t_block[1], self.y_embedder.y_proj.fc1,
                 self.y_embedder.y_proj.fc2]
        if self.micro_conditioning:
            small += [self.csize_embedder.mlp[0], self.csize_embedder.mlp[2], self.ar_embedder.mlp[0],
                      self.ar_embedder.mlp[2]]
        for m in small:
            nn.init.normal_(m.weight, std=0.02)
        for blk in self.blocks:
            nn.init.zeros_(blk.cross_attn.proj.weight)
            nn.init.zeros_(blk.cross_attn.proj.bias)
        nn.init.zeros_(self.final_layer.linear.weight)
        nn.init.zeros_(self.final_layer.linear.bias)


@MODELS.register_module()
def PixArtMS_XL_2(**kwargs):
    """PixArt-Sigma-XL/2: depth 28, width 1152, 16 heads, patch 2 (PixArtMS.py:291-293)."""
    return PixArtMS(depth=28, hidden_size=1152, patch_size=2, num_heads=16, **kwargs)


class PixArtBlock(PixArtMSBlock):
    """`PixArtBlock` of the single-scale model (nets/PixArt.py:26-57): the same adaLN-single block; `forward(x, y, t, mask)` has no HW
    argument -- the token grid is the square root of N (PixArt_blocks.py:126-127)."""

    def forward(self, x, y, t, mask=None, **kwargs):
        return super().forward(x, y, t, mask, None)


@MODELS.register_module()
class PixArt(PixArtMS):
    """Single-scale PixArt (nets/PixArt.py:62-258; registry names `PixArt`, `PixArt_XL_2`: the 256px Sigma config
    `PixArt_sigma_xl2_img256_internal.py:12`): the multi-scale model without micro-conditioning, at the fixed resolution `input_size`.
    Same state-dict keys (the frozen `pos_embed` buffer is recomputed per geometry here too; for the model's own resolution that is the
    table `initialize_weights` stores, PixArt.py:224-229), same kernels; the three forward signatures are the single-scale ones."""

    def __init__(self, input_size=32, patch_size=2, in_channels=4, hidden_size=1152, depth=28, num_heads=16, mlp_ratio=4.0,
                 class_dropout_prob=0.1, pred_sigma=True, drop_path: float = 0.0, caption_channels=4096, pe_interpolation=1.0,
                 config=None, model_max_length=120, qk_norm=False, kv_compress_config=None, **kwargs):
        super().__init__(input_size=input_size, patch_size=patch_size, in_channels=in_channels, hidden_size=hidden_size, depth=depth,
                         num_heads=num_heads, mlp_ratio=mlp_ratio, class_dropout_prob=class_dropout_prob, pred_sigma=pred_sigma,
                         drop_path=drop_path, caption_channels=caption_channels, pe_interpolation=pe_interpolation, config=config,
                         model_max_length=model_max_length, micro_condition=False, qk_norm=qk_norm,
                         kv_compress_config=kv_compress_config, **kwargs)
        self.input_size = input_size
        for blk in self.blocks:                      # same parameters and kernels, the single-scale call signature
            blk.__class__ = PixArtBlock

    def forward(self, x, timestep, y, mask=None, data_info=None, **kwargs):
        """PixArt.py:143-172: x must have the model's own resolution (the reference adds its fixed `pos_embed` table)."""
        if x.shape[-2] != self.input_size or x.shape[-1] != self.input_size:
            raise ValueError(f"PixArt is single-scale: expected {self.input_size} x {self.input_size} latents, got "
                             f"{tuple(x.shape[-2:])} (use PixArtMS for other sizes)")
        return super().forward(x, timestep, y, mask=mask, data_info=None)

    def forward_with_dpmsolver(self, x, timestep, y, mask=None, **kwargs):
        """PixArt.py:174-180."""
        return self.forward(x, timestep, y, mask).chunk(2, dim=1)[0]

    def forward_with_cfg(self, x, timestep, y, cfg_scale, mask=None, **kwargs):
        """PixArt.py:182-196 (first three channels mixed, as there)."""
        return super().forward_with_cfg(x, timestep, y, cfg_scale, None, mask=mask)


@MODELS.register_module()
def PixArt_XL_2(**kwargs):
    """PixArt-XL/2, single scale (PixArt.py:313-315)."""
    return PixArt(depth=28, hidden_size=1152, patch_size=2, num_heads=16, **kwargs)


def install_into_reference() -> bool:
    """Re-point the reference's registry and module names at these classes, so an unmodified
    `scripts/inference.py` / `train_scripts/train.py` builds the B200 model (INTEGRATION.md). Returns False when the
    reference package is not importable."""
    try:
        import diffusion.model.builder as builder          # noqa: reference package, if on sys.path
        import diffusion.model.nets as nets
    except Exception:
        return False
    for name, obj in (("PixArtMS", PixArtMS), ("PixArtMS_XL_2", PixArtMS_XL_2), ("PixArt", PixArt), ("PixArt_XL_2", PixArt_XL_2)):
        reg = builder.MODELS
        table = getattr(reg, "_module_dict", None) or getattr(reg, "module_dict", None) or getattr(reg, "_m", None)
        if table is not None:
            table[name] = obj
        setattr(nets, name, obj)
    nets.PixArtMSBlock = PixArtMSBlock
    nets.PixArtBlock = PixArtBlock
    try:                                                   # the samplers the inference script imports from `diffusion`
        import diffusion
        from .sampler import DPMS, SASolverSampler
        diffusion.DPMS = DPMS
        diffusion.SASolverSampler = SASolverSampler
    except Exception:
        pass
    return True
