"""ctypes binding of libpixart_sm100.so (the C-ABI declared in include/pixart_sm100.h).

PyTorch is used only for device memory and streams: every call passes raw `data_ptr()`s and the current
CUDA stream.  There is no fallback: if the shared library is missing or the device is not sm_100 the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PXA_LIB_PATH") or os.path.join(_HERE, "libpixart_sm100.so")   # override: experiment builds only

EPI_BIAS, EPI_BIAS_GELU, EPI_BIAS_RESIDUAL = 0, 1, 2
EPI_BIAS_GELU_AUX, EPI_MUL_DGELU = 3, 4      # MLP training fusions (include/pixart_sm100.h)
EPI_LN_BIAS, EPI_LN_BIAS_GELU = 5, 6         # fused LayerNorm-modulate consumer epilogues
LN_STAT_PARTS = 8
DTYPE_BF16, DTYPE_F32 = 0, 1


class PxaError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [("a", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p),
                ("out_aux_bf16", C.c_void_p), ("residual", C.c_void_p), ("gate", C.c_void_p),
                ("gate_batch_stride", C.c_int64), ("rows_per_batch", C.c_int32),
                ("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32),
                ("lda", C.c_int32), ("ldw", C.c_int32), ("ldo", C.c_int32),
                ("epilogue", C.c_int32), ("out_dtype", C.c_int32), ("block_n", C.c_int32), ("max_ctas", C.c_int32),
                ("cta_pair", C.c_int32), ("debug_trace", C.c_void_p), ("operands_mn_major", C.c_int32),
                ("k_splits", C.c_int32), ("aux_is_branch", C.c_int32),
                ("aux_scale", C.c_void_p), ("aux_scale_batch_stride", C.c_int64), ("row_stats_out", C.c_void_p),
                ("ln_stats", C.c_void_p), ("ln_u", C.c_void_p), ("ln_v", C.c_void_p), ("ln_uv_batch_stride", C.c_int64),
                ("ln_dim", C.c_int32), ("ln_eps", C.c_float), ("res_epilogue", C.c_int32), ("epi_warps", C.c_int32),
                ("reverse_tiles", C.c_int32)]


class LnPrepareArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("a_out", C.c_void_p), ("stats_out", C.c_void_p), ("scale", C.c_void_p),
                ("mod_batch_stride", C.c_int64), ("rows_per_batch", C.c_int32), ("M", C.c_int32), ("C", C.c_int32),
                ("ldx", C.c_int32)]


class MlpArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w1", C.c_void_p), ("b1", C.c_void_p), ("w2", C.c_void_p), ("b2", C.c_void_p), ("x32", C.c_void_p),
                ("gate", C.c_void_p), ("gate_batch_stride", C.c_int64), ("hidden_ws", C.c_void_p), ("hidden_ws_bytes", C.c_int64),
                ("flags_ws", C.c_void_p), ("flags_ws_bytes", C.c_int64), ("rows_per_batch", C.c_int32), ("M", C.c_int32),
                ("K1", C.c_int32), ("N1", C.c_int32), ("N2", C.c_int32), ("ldx", C.c_int32), ("ldw1", C.c_int32), ("ldw2", C.c_int32),
                ("ldo", C.c_int32), ("group", C.c_int32), ("ring", C.c_int32), ("max_ctas", C.c_int32), ("lag", C.c_int32), ("k_splits", C.c_int32)]


class AdamWArgs(C.Structure):
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("shadow_bf16", C.c_void_p), ("n", C.c_int64), ("step", C.c_int32), ("lr", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float), ("grad_scale", C.c_float)]


class LnModArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("out", C.c_void_p), ("shift", C.c_void_p), ("scale", C.c_void_p),
                ("mod_batch_stride", C.c_int64), ("rows_per_batch", C.c_int32),
                ("M", C.c_int32), ("C", C.c_int32), ("ldx", C.c_int32), ("x_dtype", C.c_int32), ("eps", C.c_float),
                ("reverse_rows", C.c_int32), ("max_ctas", C.c_int32)]


class AttnArgs(C.Structure):
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
                ("kv_len", C.c_void_p), ("kv_off", C.c_void_p),
                ("q_sn", C.c_int64), ("q_sh", C.c_int64),
                ("k_sn", C.c_int64), ("k_sh", C.c_int64), ("v_sn", C.c_int64), ("v_sh", C.c_int64),
                ("kv_rows", C.c_int64),
                ("B", C.c_int32), ("H", C.c_int32), ("Nq", C.c_int32), ("Nk", C.c_int32),
                ("ldo", C.c_int32), ("scale", C.c_float), ("debug_trace", C.c_void_p), ("lse", C.c_void_p),
                ("reverse_batch", C.c_int32), ("variant", C.c_int32), ("p_precision", C.c_int32), ("reserved0", C.c_int32)]


class T5AttnArgs(C.Structure):
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p), ("bias", C.c_void_p),
                ("key_bias", C.c_void_p), ("q_sn", C.c_int64), ("q_sh", C.c_int64), ("k_sn", C.c_int64), ("k_sh", C.c_int64),
                ("v_sn", C.c_int64), ("v_sh", C.c_int64), ("ldo", C.c_int64), ("B", C.c_int32), ("H", C.c_int32), ("L", C.c_int32),
                ("scale", C.c_float), ("rel_bias", C.c_void_p)]


class KvCompressArgs(C.Structure):
    _fields_ = [("k_in", C.c_void_p), ("v_in", C.c_void_p), ("k_out", C.c_void_p), ("v_out", C.c_void_p),
                ("conv_w", C.c_void_p), ("conv_b", C.c_void_p), ("ln_w", C.c_void_p), ("ln_b", C.c_void_p),
                ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32), ("ld_in", C.c_int32),
                ("eps", C.c_float)]


class Conv3x3Args(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p), ("residual", C.c_void_p),
                ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("Cin", C.c_int32), ("Cout", C.c_int32)]


class DpmStepArgs(C.Structure):
    _fields_ = [("model_out", C.c_void_p), ("x", C.c_void_p), ("x0_prev", C.c_void_p), ("out_batch_stride", C.c_int64),
                ("n", C.c_int32), ("hw", C.c_int32), ("out_dtype", C.c_int32),
                ("cfg_scale", C.c_float), ("sigma_s", C.c_float), ("inv_alpha_s", C.c_float),
                ("a", C.c_float), ("b", C.c_float), ("c", C.c_float)]


class SaStepArgs(C.Structure):
    _fields_ = [("model_out", C.c_void_p), ("x", C.c_void_p), ("x_pred", C.c_void_p), ("x0_prev", C.c_void_p),
                ("noise", C.c_void_p), ("noise_next", C.c_void_p), ("out_batch_stride", C.c_int64),
                ("n", C.c_int32), ("hw", C.c_int32), ("cond_row_offset", C.c_int32), ("out_dtype", C.c_int32),
                ("has_corr", C.c_int32), ("cfg_scale", C.c_float), ("sigma", C.c_float), ("inv_alpha", C.c_float),
                ("cA", C.c_float), ("c0", C.c_float), ("c1", C.c_float), ("cN", C.c_float),
                ("pA", C.c_float), ("p0", C.c_float), ("p1", C.c_float), ("pN", C.c_float)]


class GateResidualArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("y", C.c_void_p), ("gate", C.c_void_p), ("out", C.c_void_p), ("dgate", C.c_void_p),
                ("gate_batch_stride", C.c_int64), ("rows_per_batch", C.c_int32), ("M", C.c_int32), ("C", C.c_int32)]


class LnModBwdArgs(C.Structure):
    _fields_ = [("x", C.c_void_p), ("dxn", C.c_void_p), ("scale", C.c_void_p), ("dx", C.c_void_p), ("dshift", C.c_void_p),
                ("dscale", C.c_void_p), ("mod_batch_stride", C.c_int64), ("rows_per_batch", C.c_int32),
                ("M", C.c_int32), ("C", C.c_int32), ("eps", C.c_float), ("add_in", C.c_void_p)]


class KvCompressBwdArgs(C.Structure):
    _fields_ = [("k_in", C.c_void_p), ("v_in", C.c_void_p), ("dk_out", C.c_void_p), ("dv_out", C.c_void_p),
                ("dk_in", C.c_void_p), ("dv_in", C.c_void_p), ("conv_w", C.c_void_p), ("conv_b", C.c_void_p),
                ("ln_w", C.c_void_p), ("d_conv_w", C.c_void_p), ("d_conv_b", C.c_void_p), ("d_ln_w", C.c_void_p),
                ("d_ln_b", C.c_void_p), ("B", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32),
                ("ld_in", C.c_int32), ("ld_din", C.c_int32), ("eps", C.c_float)]


class AttnBwdArgs(C.Structure):
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("o", C.c_void_p), ("d_o", C.c_void_p),
                ("lse", C.c_void_p), ("delta", C.c_void_p), ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p),
                ("kv_len", C.c_void_p), ("kv_off", C.c_void_p),
                ("q_sn", C.c_int64), ("q_sh", C.c_int64), ("k_sn", C.c_int64), ("k_sh", C.c_int64),
                ("v_sn", C.c_int64), ("v_sh", C.c_int64),
                ("dq_sn", C.c_int64), ("dq_sh", C.c_int64), ("dk_sn", C.c_int64), ("dk_sh", C.c_int64),
                ("dv_sn", C.c_int64), ("dv_sh", C.c_int64),
                ("ldo", C.c_int64), ("lddo", C.c_int64), ("kv_rows", C.c_int64),
                ("B", C.c_int32), ("H", C.c_int32), ("Nq", C.c_int32), ("Nk", C.c_int32), ("scale", C.c_float)]


EXPORTS = ("pxa_transpose_bf16", "pxa_gelu_tanh_bf16", "pxa_gate_residual_fwd", "pxa_gate_residual_bwd",
           "pxa_ln_modulate_bwd", "pxa_colsum_bf16", "pxa_attn_delta_d72", "pxa_flash_attn_d72_bwd_bf16", "pxa_kv_compress_conv2_ln_bwd",
           "pxa_version", "pxa_last_error", "pxa_launch_count", "pxa_gemm_bf16", "pxa_ln_modulate",
           "pxa_flash_attn_d72_bf16", "pxa_kv_compress_conv2_ln", "pxa_conv3x3_nhwc_bf16", "pxa_dpm_solver_pp_step",
           "pxa_ln_prepare", "pxa_layernorm_affine_bf16", "pxa_groupnorm_silu_nhwc_bf16", "pxa_adamw_flat", "pxa_mlp_fused_bf16",
           "pxa_rmsnorm_bf16", "pxa_t5_attn_d64_bf16", "pxa_sa_solver_step")

_lib = None


def load() -> C.CDLL:
    """Load the C-ABI library (built in-tree by `pixart_sigma_b200.build`). Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PxaError(f"{LIB_PATH} not found: run `python -m pixart_sigma_b200.build` (there is no fallback path)")
        lib = C.CDLL(LIB_PATH)
        lib.pxa_version.restype = C.c_int
        lib.pxa_last_error.restype = C.c_char_p
        lib.pxa_launch_count.restype = C.c_uint64
        for name, struct in (("pxa_gemm_bf16", GemmArgs), ("pxa_ln_modulate", LnModArgs),
                             ("pxa_flash_attn_d72_bf16", AttnArgs), ("pxa_kv_compress_conv2_ln", KvCompressArgs),
                             ("pxa_conv3x3_nhwc_bf16", Conv3x3Args), ("pxa_dpm_solver_pp_step", DpmStepArgs),
                             ("pxa_sa_solver_step", SaStepArgs), ("pxa_ln_prepare", LnPrepareArgs), ("pxa_adamw_flat", AdamWArgs),
                             ("pxa_mlp_fused_bf16", MlpArgs), ("pxa_t5_attn_d64_bf16", T5AttnArgs)):
            fn = getattr(lib, name)
            fn.restype = C.c_int
            fn.argtypes = [C.POINTER(struct), C.c_void_p]
        for name, struct in (("pxa_gate_residual_fwd", GateResidualArgs), ("pxa_gate_residual_bwd", GateResidualArgs),
                             ("pxa_ln_modulate_bwd", LnModBwdArgs), ("pxa_flash_attn_d72_bwd_bf16", AttnBwdArgs),
                             ("pxa_kv_compress_conv2_ln_bwd", KvCompressBwdArgs)):
            fn = getattr(lib, name)
            fn.restype = C.c_int
            fn.argtypes = [C.POINTER(struct), C.c_void_p]
        lib.pxa_layernorm_affine_bf16.restype = C.c_int
        lib.pxa_layernorm_affine_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_float,
                                                  C.c_void_p]
        lib.pxa_rmsnorm_bf16.restype = C.c_int
        lib.pxa_rmsnorm_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_float,
                                         C.c_void_p]
        lib.pxa_groupnorm_silu_nhwc_bf16.restype = C.c_int
        lib.pxa_groupnorm_silu_nhwc_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                                     C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_void_p]
        lib.pxa_transpose_bf16.restype = C.c_int
        lib.pxa_transpose_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_void_p]
        lib.pxa_gelu_tanh_bf16.restype = C.c_int
        lib.pxa_gelu_tanh_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        lib.pxa_colsum_bf16.restype = C.c_int
        lib.pxa_colsum_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_void_p]
        lib.pxa_attn_delta_d72.restype = C.c_int
        lib.pxa_attn_delta_d72.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                                           C.c_int64, C.c_void_p]
        _lib = lib
    return _lib


def launch_count() -> int:
    return int(load().pxa_launch_count())


def _check(rc: int, what: str) -> None:
    if rc != 0:
        raise PxaError(f"{what} failed ({rc}): {load().pxa_last_error().decode()}")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _dt(dtype: torch.dtype) -> int:
    if dtype == torch.bfloat16:
        return DTYPE_BF16
    if dtype == torch.float32:
        return DTYPE_F32
    raise PxaError(f"unsupported dtype {dtype}")


def gemm(a: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor, *,
         epilogue: int = EPI_BIAS, residual: Optional[torch.Tensor] = None, gate: Optional[torch.Tensor] = None,
         gate_batch_stride: int = 0, rows_per_batch: int = 0, out_aux: Optional[torch.Tensor] = None,
         block_n: int = 0, max_ctas: int = 0, cta_pair: int = 0, debug_trace: Optional[torch.Tensor] = None,
         aux_is_branch: bool = False, aux_scale: Optional[torch.Tensor] = None, aux_scale_batch_stride: int = 0,
         row_stats_out: Optional[torch.Tensor] = None, ln_stats: Optional[torch.Tensor] = None,
         ln_u: Optional[torch.Tensor] = None, ln_v: Optional[torch.Tensor] = None, ln_uv_batch_stride: int = 0,
         ln_dim: int = 0, ln_eps: float = 1e-6, res_epilogue: int = 0, epi_warps: int = 0,
         reverse_tiles: bool = False) -> torch.Tensor:
    """out = epilogue(a @ w.T + bias). a (M,K) bf16, w (N,K) bf16 (nn.Linear layout), both K-contiguous.

    Fused LayerNorm-modulate (include/pixart_sm100.h, PXA_EPI_LN_BIAS): the fp32 residual epilogue can emit the scaled bf16
    copy `out_aux = out * aux_scale[b]` and the per-row partial sums `row_stats_out` (M, 8, 2); the EPI_LN_* epilogues
    consume them (`ln_stats`) together with the per-sample vectors `ln_u`, `ln_v` (fp32 views, row b at b * stride)."""
    assert a.is_cuda and a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1 and out.dim() == 2 and out.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K and out.shape == (M, N)
    if bias is not None:
        assert bias.dtype == torch.bfloat16 and bias.is_contiguous() and bias.numel() == N
    if residual is not None:
        assert residual.dtype == out.dtype and residual.shape == out.shape and residual.stride() == out.stride()
    if gate is not None:
        assert gate.dtype == torch.float32
    if out_aux is not None:
        assert out_aux.dtype == torch.bfloat16 and out_aux.shape == out.shape and out_aux.stride() == out.stride()
    for tns in (aux_scale, ln_u, ln_v):
        assert tns is None or (tns.dtype == torch.float32 and tns.is_cuda)
    for tns in (row_stats_out, ln_stats):
        assert tns is None or (tns.dtype == torch.float32 and tns.is_contiguous() and tns.numel() == M * LN_STAT_PARTS * 2)
    args = GemmArgs(a=_ptr(a), w=_ptr(w), bias=_ptr(bias), out=_ptr(out), out_aux_bf16=_ptr(out_aux),
                    residual=_ptr(residual), gate=_ptr(gate), gate_batch_stride=gate_batch_stride,
                    rows_per_batch=rows_per_batch or M, M=M, N=N, K=K, lda=a.stride(0), ldw=w.stride(0),
                    ldo=out.stride(0), epilogue=epilogue, out_dtype=_dt(out.dtype), block_n=block_n, max_ctas=max_ctas,
                    cta_pair=cta_pair, debug_trace=_ptr(debug_trace), operands_mn_major=0, k_splits=0,
                    aux_is_branch=int(aux_is_branch), aux_scale=_ptr(aux_scale), aux_scale_batch_stride=aux_scale_batch_stride,
                    row_stats_out=_ptr(row_stats_out), ln_stats=_ptr(ln_stats), ln_u=_ptr(ln_u), ln_v=_ptr(ln_v),
                    ln_uv_batch_stride=ln_uv_batch_stride, ln_dim=ln_dim, ln_eps=ln_eps, res_epilogue=res_epilogue,
                    epi_warps=epi_warps, reverse_tiles=int(reverse_tiles))
    _check(load().pxa_gemm_bf16(C.byref(args), _stream()), "pxa_gemm_bf16")
    return out


def ln_prepare(x: torch.Tensor, mult: torch.Tensor, a_out: torch.Tensor, stats_out: torch.Tensor, *, mod_batch_stride: int,
               rows_per_batch: int) -> None:
    """First link of the fused LayerNorm-modulate chain: a_out = bf16(x * mult[b]) with mult = 1 + scale (the multiplier
    `gemm(aux_scale=...)` takes), stats_out (M, 8, 2) = partial (sum, sum of squares) of each row of x (part 0; the rest
    zero).  x (M, C) fp32, mult an fp32 view (row b at b*stride)."""
    scale = mult
    assert x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1 and scale.dtype == torch.float32
    M, Cc = x.shape
    assert a_out.dtype == torch.bfloat16 and a_out.is_contiguous() and a_out.shape == (M, Cc)
    assert stats_out.dtype == torch.float32 and stats_out.is_contiguous() and stats_out.numel() == M * LN_STAT_PARTS * 2
    args = LnPrepareArgs(x=_ptr(x), a_out=_ptr(a_out), stats_out=_ptr(stats_out), scale=_ptr(scale),
                         mod_batch_stride=mod_batch_stride, rows_per_batch=rows_per_batch, M=M, C=Cc, ldx=x.stride(0))
    _check(load().pxa_ln_prepare(C.byref(args), _stream()), "pxa_ln_prepare")


def ln_modulate(x: torch.Tensor, shift: torch.Tensor, scale: torch.Tensor, out: torch.Tensor, *,
                mod_batch_stride: int, rows_per_batch: int, eps: float = 1e-6, reverse_rows: bool = False,
                max_ctas: int = 0) -> torch.Tensor:
    """out = LN(x) * (1 + scale[b]) + shift[b]; x (M,C) fp32/bf16, shift/scale fp32 views (row b at b*stride)."""
    assert x.dim() == 2 and x.stride(1) == 1 and out.is_contiguous() and out.dtype == torch.bfloat16
    assert shift.dtype == torch.float32 and scale.dtype == torch.float32
    M, Cc = x.shape
    args = LnModArgs(x=_ptr(x), out=_ptr(out), shift=_ptr(shift), scale=_ptr(scale), mod_batch_stride=mod_batch_stride,
                     rows_per_batch=rows_per_batch, M=M, C=Cc, ldx=x.stride(0), x_dtype=_dt(x.dtype), eps=eps,
                     reverse_rows=int(reverse_rows), max_ctas=max_ctas)
    _check(load().pxa_ln_modulate(C.byref(args), _stream()), "pxa_ln_modulate")
    return out


_ATTN_VARIANT = int(os.environ.get("PXA_ATTN_VARIANT", "0"))      # A/B switch for the attention forward (0 = library default)


def layernorm_affine_(x: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor, eps: float = 1e-5) -> torch.Tensor:
    """In-place LayerNorm with affine parameters on the rows of a bf16 (M, 1152) view with unit column stride (qk_norm)."""
    assert x.dtype == weight.dtype == bias.dtype == torch.bfloat16 and x.dim() == 2 and x.stride(1) == 1
    assert weight.is_contiguous() and bias.is_contiguous() and weight.numel() == bias.numel() == x.shape[1]
    _check(load().pxa_layernorm_affine_bf16(_ptr(x), _ptr(weight), _ptr(bias), x.shape[0], x.shape[1], x.stride(0), eps,
                                            _stream()), "pxa_layernorm_affine_bf16")
    return x


def rmsnorm(x: torch.Tensor, weight: torch.Tensor, out: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """T5LayerNorm: out (M, C) bf16 = x * rsqrt(mean(x^2) + eps) * weight on the rows of the fp32 stream x (M, C)."""
    assert x.is_cuda and x.dtype == torch.float32 and out.dtype == weight.dtype == torch.bfloat16
    assert x.dim() == 2 and out.shape == x.shape and x.stride(1) == 1 and out.stride(1) == 1
    assert weight.is_contiguous() and weight.numel() == x.shape[1]
    _check(load().pxa_rmsnorm_bf16(_ptr(x), _ptr(weight), _ptr(out), x.shape[0], x.shape[1], x.stride(0), out.stride(0), eps,
                                   _stream()), "pxa_rmsnorm_bf16")
    return out


T5_ATTN_MAX_KEYS = 384


def t5_attn(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, bias: Optional[torch.Tensor],
            key_bias: Optional[torch.Tensor] = None, *, B: int, H: int, L: int, scale: float = 1.0,
            rel_bias: Optional[torch.Tensor] = None) -> torch.Tensor:
    """T5 self-attention, head_dim 64, L <= 384: out (B*L, H*64) = softmax(q k^T * scale + bias[h] + key_bias[b]) v.
    q / k / v: bf16 (B*L, H*64) views with unit column stride (e.g. column slices of a fused qkv GEMM output);
    bias fp32 (H, L, L), or rel_bias fp32 (H, 2L-1) with bias[h, i, j] = rel_bias[h, j - i + L - 1]; key_bias fp32 (B, L) or None."""
    for t in (q, k, v, out):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.dim() == 2 and t.stride(1) == 1 and t.shape == (B * L, H * 64)
    assert (bias is None) != (rel_bias is None), "exactly one of bias / rel_bias"
    assert bias is None or (bias.dtype == torch.float32 and bias.is_contiguous() and bias.shape == (H, L, L))
    assert rel_bias is None or (rel_bias.dtype == torch.float32 and rel_bias.is_contiguous() and rel_bias.shape == (H, 2 * L - 1))
    assert key_bias is None or (key_bias.dtype == torch.float32 and key_bias.is_contiguous() and key_bias.shape == (B, L))
    args = T5AttnArgs(q=_ptr(q), k=_ptr(k), v=_ptr(v), out=_ptr(out), bias=_ptr(bias), key_bias=_ptr(key_bias),
                      q_sn=q.stride(0), q_sh=64, k_sn=k.stride(0), k_sh=64, v_sn=v.stride(0), v_sh=64, ldo=out.stride(0),
                      B=B, H=H, L=L, scale=scale, rel_bias=_ptr(rel_bias))
    _check(load().pxa_t5_attn_d64_bf16(C.byref(args), _stream()), "pxa_t5_attn_d64_bf16")
    return out


def flash_attn(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, *, B: int, H: int, Nq: int,
               Nk: int, kv_rows: int, kv_len: Optional[torch.Tensor] = None, kv_off: Optional[torch.Tensor] = None,
               q_strides=None, k_strides=None, v_strides=None, scale: Optional[float] = None,
               debug_trace: Optional[torch.Tensor] = None, lse: Optional[torch.Tensor] = None,
               variant: int = 0, reverse_batch: bool = False, fp32_p: bool = False) -> torch.Tensor:
    """Head-dim-72 attention. q/k/v are bf16 *views*; strides are (row, head) in elements, e.g. slices of the
    (rows, 3, H, 72) qkv GEMM output. out is (B*Nq, H*72) bf16.  fp32_p: `fp32_attention` grade P V (P as bf16 hi + lo)."""
    assert q.dtype == k.dtype == v.dtype == out.dtype == torch.bfloat16
    for tns in (kv_len, kv_off):
        if tns is not None:
            assert tns.dtype == torch.int32 and tns.is_cuda and tns.numel() == B
    args = AttnArgs(q=_ptr(q), k=_ptr(k), v=_ptr(v), out=_ptr(out), kv_len=_ptr(kv_len), kv_off=_ptr(kv_off),
                    q_sn=q_strides[0], q_sh=q_strides[1], k_sn=k_strides[0], k_sh=k_strides[1],
                    v_sn=v_strides[0], v_sh=v_strides[1], kv_rows=kv_rows, B=B, H=H, Nq=Nq, Nk=Nk,
                    ldo=out.stride(0), scale=scale if scale is not None else 72 ** -0.5,
                    debug_trace=_ptr(debug_trace), lse=_ptr(lse), variant=variant or _ATTN_VARIANT,
                    reverse_batch=int(reverse_batch), p_precision=int(bool(fp32_p)), reserved0=0)
    if lse is not None:
        assert lse.dtype == torch.float32 and lse.is_contiguous() and lse.numel() == B * H * Nq
    _check(load().pxa_flash_attn_d72_bf16(C.byref(args), _stream()), "pxa_flash_attn_d72_bf16")
    return out


def kv_compress(k_in: torch.Tensor, v_in: torch.Tensor, k_out: torch.Tensor, v_out: torch.Tensor, conv_w, conv_b,
                ln_w, ln_b, *, B: int, H: int, W: int, ld_in: int, eps: float = 1e-5) -> None:
    args = KvCompressArgs(k_in=_ptr(k_in), v_in=_ptr(v_in), k_out=_ptr(k_out), v_out=_ptr(v_out), conv_w=_ptr(conv_w),
                          conv_b=_ptr(conv_b), ln_w=_ptr(ln_w), ln_b=_ptr(ln_b), B=B, H=H, W=W, C=k_out.shape[-1],
                          ld_in=ld_in, eps=eps)
    _check(load().pxa_kv_compress_conv2_ln(C.byref(args), _stream()), "pxa_kv_compress_conv2_ln")


def conv3x3_nhwc(x: torch.Tensor, w_packed: torch.Tensor, bias: Optional[torch.Tensor], out: torch.Tensor,
                 residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """3x3 / stride 1 / pad 1 convolution on NHWC bf16 tensors. x (B,H,W,Cin), w_packed (Cout,3,3,Cin), out (B,H,W,Cout)."""
    assert x.dtype == w_packed.dtype == out.dtype == torch.bfloat16 and x.is_contiguous() and w_packed.is_contiguous()
    assert out.is_contiguous() and (residual is None or (residual.is_contiguous() and residual.shape == out.shape))
    B, H, W, Cin = x.shape
    Cout = w_packed.shape[0]
    assert w_packed.shape == (Cout, 3, 3, Cin) and out.shape == (B, H, W, Cout)
    args = Conv3x3Args(x=_ptr(x), w=_ptr(w_packed), bias=_ptr(bias), out=_ptr(out), residual=_ptr(residual), B=B, H=H, W=W,
                       Cin=Cin, Cout=Cout)
    _check(load().pxa_conv3x3_nhwc_bf16(C.byref(args), _stream()), "pxa_conv3x3_nhwc_bf16")
    return out


def _env_int(name: str, default: int) -> int:
    return int(os.environ.get(name, default))


# fc2 trails fc1 by LAG groups of GROUP 256-row panels; the ring holds RING = LAG + 2 groups (mlp_sm100.cu)
MLP_GROUP, MLP_LAG = _env_int("PXA_MLP_GROUP", 4), _env_int("PXA_MLP_LAG", 1)
MLP_RING = _env_int("PXA_MLP_RING", MLP_LAG + 2)


def mlp_fused_workspace(M: int, n_hidden: int, device, group: int = MLP_GROUP, ring: int = MLP_RING):
    """(hidden ring, flag array) for `mlp_fused` at M rows."""
    panels = (M + 255) // 256
    hidden = torch.empty(ring * group * 256 * n_hidden, dtype=torch.bfloat16, device=device)
    flags = torch.empty(2 * panels + (panels + group - 1) // group + 4, dtype=torch.int32, device=device)
    return hidden, flags


def mlp_fused(x: torch.Tensor, w1: torch.Tensor, b1: Optional[torch.Tensor], w2: torch.Tensor, b2: Optional[torch.Tensor],
              x32: torch.Tensor, *, gate: Optional[torch.Tensor] = None, gate_batch_stride: int = 0, rows_per_batch: int = 0,
              hidden_ws: torch.Tensor, flags_ws: torch.Tensor, group: int = MLP_GROUP, ring: int = MLP_RING, lag: int = MLP_LAG,
              max_ctas: int = 0, k_splits: int = 0) -> torch.Tensor:
    """x32 += gate[b] * (gelu_tanh(x @ w1.T + b1) @ w2.T + b2) in ONE persistent kernel (include/pixart_sm100.h, PxaMlpArgs)."""
    assert x.dtype == w1.dtype == w2.dtype == torch.bfloat16 and x32.dtype == torch.float32 and x.is_cuda
    assert x.dim() == 2 and x.stride(1) == 1 and w1.stride(1) == 1 and w2.stride(1) == 1 and x32.stride(1) == 1
    M, K1 = x.shape
    N1, N2 = w1.shape[0], w2.shape[0]
    assert w1.shape[1] == K1 and w2.shape[1] == N1 and x32.shape == (M, N2)
    assert hidden_ws.dtype == torch.bfloat16 and hidden_ws.is_contiguous() and flags_ws.dtype == torch.int32 and flags_ws.is_contiguous()
    args = MlpArgs(x=_ptr(x), w1=_ptr(w1), b1=_ptr(b1), w2=_ptr(w2), b2=_ptr(b2), x32=_ptr(x32), gate=_ptr(gate),
                   gate_batch_stride=gate_batch_stride, hidden_ws=_ptr(hidden_ws), hidden_ws_bytes=hidden_ws.numel() * 2,
                   flags_ws=_ptr(flags_ws), flags_ws_bytes=flags_ws.numel() * 4, rows_per_batch=rows_per_batch or M, M=M, K1=K1,
                   N1=N1, N2=N2, ldx=x.stride(0), ldw1=w1.stride(0), ldw2=w2.stride(0), ldo=x32.stride(0), group=group, ring=ring,
                   max_ctas=max_ctas, lag=lag, k_splits=k_splits)
    _check(load().pxa_mlp_fused_bf16(C.byref(args), _stream()), "pxa_mlp_fused_bf16")
    return x32


def adamw_flat(param: torch.Tensor, grad: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, *, step: int, lr: float,
               betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2, grad_scale: float = 1.0,
               shadow: Optional[torch.Tensor] = None) -> None:
    """torch.optim.AdamW's update on flat fp32 tensors of equal length (a multiple of 4), in place; `shadow` (bf16, same
    length) receives the bf16 copy of the new parameters."""
    for t in (param, grad, exp_avg, exp_avg_sq):
        assert t.dtype == torch.float32 and t.is_cuda and t.is_contiguous() and t.numel() == param.numel()
    assert shadow is None or (shadow.dtype == torch.bfloat16 and shadow.is_contiguous() and shadow.numel() == param.numel())
    args = AdamWArgs(param=_ptr(param), grad=_ptr(grad), exp_avg=_ptr(exp_avg), exp_avg_sq=_ptr(exp_avg_sq), shadow_bf16=_ptr(shadow),
                     n=param.numel(), step=step, lr=lr, beta1=betas[0], beta2=betas[1], eps=eps, weight_decay=weight_decay,
                     grad_scale=grad_scale)
    _check(load().pxa_adamw_flat(C.byref(args), _stream()), "pxa_adamw_flat")


def groupnorm_silu_nhwc(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, out: torch.Tensor, *, groups: int = 32,
                        eps: float = 1e-6, silu: bool = True, stats_ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GroupNorm (+ SiLU) on an NHWC bf16 image x (B, H, W, C) -> out (same shape); statistics in fp32."""
    assert x.dtype == out.dtype == gamma.dtype == beta.dtype == torch.bfloat16 and x.is_contiguous() and out.is_contiguous()
    B, H, W, Cc = x.shape
    assert out.shape == x.shape and gamma.numel() == beta.numel() == Cc and gamma.is_contiguous() and beta.is_contiguous()
    if stats_ws is None:
        stats_ws = torch.empty(B * groups * 2, dtype=torch.float32, device=x.device)
    assert stats_ws.dtype == torch.float32 and stats_ws.numel() >= B * groups * 2
    _check(load().pxa_groupnorm_silu_nhwc_bf16(_ptr(x), _ptr(out), _ptr(gamma), _ptr(beta), _ptr(stats_ws), B, H * W, Cc, groups,
                                               eps, int(silu), _stream()), "pxa_groupnorm_silu_nhwc_bf16")
    return out


def dpm_solver_pp_step(model_out: torch.Tensor, x: torch.Tensor, x0_prev: torch.Tensor, *, cfg_scale: float, sigma_s: float,
                       alpha_s: float, a: float, b: float, c: float) -> torch.Tensor:
    """One DPM-Solver++ (2M) update, in place on x and x0_prev (include/pixart_sm100.h: pxa_dpm_solver_pp_step).
    model_out: denoiser output of the CFG batch [uncond; cond], (2n, C>=4, h, w) fp32 or bf16 -- a channel-sliced view of
    the 8-channel learn-sigma output is fine; x, x0_prev: fp32 (n, 4, h, w) contiguous."""
    assert model_out.is_cuda and x.is_cuda and x0_prev.is_cuda and x.dtype == x0_prev.dtype == torch.float32
    assert x.is_contiguous() and x0_prev.is_contiguous() and x.shape == x0_prev.shape and x.dim() == 4 and x.shape[1] == 4
    n, _, h, w = x.shape
    assert model_out.shape[0] == 2 * n and model_out.shape[1] >= 4 and model_out.shape[2:] == (h, w)
    assert model_out.stride(3) == 1 and model_out.stride(2) == w and model_out.stride(1) == h * w, "model_out: (.., h, w) planes must be dense"
    args = DpmStepArgs(model_out=_ptr(model_out), x=_ptr(x), x0_prev=_ptr(x0_prev), out_batch_stride=model_out.stride(0),
                       n=n, hw=h * w, out_dtype=_dt(model_out.dtype), cfg_scale=cfg_scale, sigma_s=sigma_s,
                       inv_alpha_s=1.0 / alpha_s, a=a, b=b, c=c)
    _check(load().pxa_dpm_solver_pp_step(C.byref(args), _stream()), "pxa_dpm_solver_pp_step")
    return x


def sa_solver_step(model_out: torch.Tensor, x: torch.Tensor, x_pred: torch.Tensor, x0_prev: torch.Tensor, noise: torch.Tensor,
                   noise_next: torch.Tensor, *, guided: bool, cfg_scale: float, sigma: float, inv_alpha: float, has_corr: bool,
                   cA: float, c0: float, c1: float, cN: float, pA: float, p0: float, p1: float, pN: float) -> torch.Tensor:
    """One SA-Solver evaluation step (corrector of step i, predictor of step i + 1), in place on x, x_pred and x0_prev
    (include/pixart_sm100.h: pxa_sa_solver_step).  model_out: denoiser output, (2n, C>=4, h, w) [uncond; cond] when guided,
    else (n, C>=4, h, w), fp32 or bf16 -- a channel-sliced view of the 8-channel learn-sigma output is fine; the state and
    noise tensors: fp32 (n, 4, h, w) contiguous."""
    for t in (x, x_pred, x0_prev, noise, noise_next):
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == x.shape
    assert model_out.is_cuda and x.dim() == 4 and x.shape[1] == 4
    n, _, h, w = x.shape
    assert model_out.shape[0] == (2 * n if guided else n) and model_out.shape[1] >= 4 and model_out.shape[2:] == (h, w)
    assert model_out.stride(3) == 1 and model_out.stride(2) == w and model_out.stride(1) == h * w, "model_out: (.., h, w) planes must be dense"
    args = SaStepArgs(model_out=_ptr(model_out), x=_ptr(x), x_pred=_ptr(x_pred), x0_prev=_ptr(x0_prev), noise=_ptr(noise),
                      noise_next=_ptr(noise_next), out_batch_stride=model_out.stride(0), n=n, hw=h * w,
                      cond_row_offset=n if guided else 0, out_dtype=_dt(model_out.dtype), has_corr=int(bool(has_corr)),
                      cfg_scale=cfg_scale, sigma=sigma, inv_alpha=inv_alpha, cA=cA, c0=c0, c1=c1, cN=cN, pA=pA, p0=p0,
                      p1=p1, pN=pN)
    _check(load().pxa_sa_solver_step(C.byref(args), _stream()), "pxa_sa_solver_step")
    return x_pred


# ------------------------------------------------------------------------------------------------- training backward
def transpose(a: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out (C, R) = a (R, C)^T, bf16; a may be a row-strided view (e.g. a column slice)."""
    assert a.dtype == torch.bfloat16 and a.dim() == 2 and a.stride(1) == 1
    R, Cc = a.shape
    if out is None:
        out = torch.empty((Cc, R), dtype=torch.bfloat16, device=a.device)
    assert out.shape == (Cc, R) and out.stride(1) == 1
    _check(load().pxa_transpose_bf16(_ptr(a), _ptr(out), R, Cc, a.stride(0), out.stride(0), _stream()), "pxa_transpose_bf16")
    return out


def gelu_tanh(pre: torch.Tensor, out: Optional[torch.Tensor] = None, dh: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dh None: out = gelu_tanh(pre); else out = dh * gelu_tanh'(pre). Contiguous bf16 tensors."""
    assert pre.dtype == torch.bfloat16 and pre.is_contiguous()
    if out is None:
        out = torch.empty_like(pre)
    assert out.is_contiguous() and out.dtype == torch.bfloat16 and (dh is None or (dh.is_contiguous() and dh.dtype == torch.bfloat16))
    _check(load().pxa_gelu_tanh_bf16(_ptr(pre), _ptr(dh), _ptr(out), pre.numel(), _stream()), "pxa_gelu_tanh_bf16")
    return out


def gate_residual_fwd(x: torch.Tensor, y: torch.Tensor, gate: Optional[torch.Tensor], out: torch.Tensor, *,
                      gate_batch_stride: int = 0, rows_per_batch: int = 0) -> torch.Tensor:
    """out = x + gate[b] * y on the fp32 residual stream (x, out fp32 (M, C); y bf16; gate fp32 view or None)."""
    assert x.dtype == out.dtype == torch.float32 and y.dtype == torch.bfloat16
    assert x.is_contiguous() and y.is_contiguous() and out.is_contiguous() and x.shape == y.shape == out.shape
    M, Cc = x.shape
    args = GateResidualArgs(x=_ptr(x), y=_ptr(y), gate=_ptr(gate), out=_ptr(out), dgate=None,
                            gate_batch_stride=gate_batch_stride, rows_per_batch=rows_per_batch or M, M=M, C=Cc)
    _check(load().pxa_gate_residual_fwd(C.byref(args), _stream()), "pxa_gate_residual_fwd")
    return out


def gate_residual_bwd(dout: torch.Tensor, y: Optional[torch.Tensor], gate: Optional[torch.Tensor], dy: torch.Tensor,
                      dgate: Optional[torch.Tensor], *, gate_batch_stride: int = 0, rows_per_batch: int = 0) -> torch.Tensor:
    """dy = bf16(dout * gate[b]); dgate[b] += sum_rows dout * y (dgate fp32 (B, C) contiguous, pre-zeroed by the caller)."""
    assert dout.dtype == torch.float32 and dout.is_contiguous() and dy.dtype == torch.bfloat16 and dy.is_contiguous()
    assert dgate is None or (dgate.dtype == torch.float32 and dgate.is_contiguous() and y is not None and y.is_contiguous())
    M, Cc = dout.shape
    args = GateResidualArgs(x=_ptr(dout), y=_ptr(y), gate=_ptr(gate), out=_ptr(dy), dgate=_ptr(dgate),
                            gate_batch_stride=gate_batch_stride, rows_per_batch=rows_per_batch or M, M=M, C=Cc)
    _check(load().pxa_gate_residual_bwd(C.byref(args), _stream()), "pxa_gate_residual_bwd")
    return dy


def ln_modulate_bwd(x: torch.Tensor, dxn: torch.Tensor, scale: torch.Tensor, dx: torch.Tensor, dshift: torch.Tensor,
                    dscale: torch.Tensor, *, mod_batch_stride: int, rows_per_batch: int, eps: float = 1e-6,
                    add_in: Optional[torch.Tensor] = None) -> None:
    """Backward of ln_modulate: dx written (= add_in + the gradient through the norm when add_in is given; add_in may be dx
    itself), dshift / dscale (B, C) fp32 accumulated."""
    assert add_in is None or (add_in.dtype == torch.float32 and add_in.is_contiguous() and add_in.shape == x.shape)
    assert x.dtype == dx.dtype == torch.float32 and dxn.dtype == torch.bfloat16
    assert x.is_contiguous() and dxn.is_contiguous() and dx.is_contiguous() and dshift.is_contiguous() and dscale.is_contiguous()
    assert dshift.dtype == dscale.dtype == scale.dtype == torch.float32
    M, Cc = x.shape
    args = LnModBwdArgs(x=_ptr(x), dxn=_ptr(dxn), scale=_ptr(scale), dx=_ptr(dx), dshift=_ptr(dshift), dscale=_ptr(dscale),
                        mod_batch_stride=mod_batch_stride, rows_per_batch=rows_per_batch, M=M, C=Cc, eps=eps,
                        add_in=_ptr(add_in))
    _check(load().pxa_ln_modulate_bwd(C.byref(args), _stream()), "pxa_ln_modulate_bwd")


def colsum(a: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """out[c] += sum_r a[r, c]; a bf16 (M, N) row-strided view, out fp32 (N,)."""
    assert a.dtype == torch.bfloat16 and a.dim() == 2 and a.stride(1) == 1 and out.dtype == torch.float32 and out.is_contiguous()
    M, N = a.shape
    assert out.numel() == N
    _check(load().pxa_colsum_bf16(_ptr(a), _ptr(out), M, N, a.stride(0), _stream()), "pxa_colsum_bf16")
    return out


def flash_attn_bwd(q, k, v, o, d_o, lse, dq, dk, dv, *, B: int, H: int, Nq: int, Nk: int, kv_rows: int,
                   kv_len: Optional[torch.Tensor] = None, kv_off: Optional[torch.Tensor] = None, q_strides, k_strides,
                   v_strides, dq_strides, dk_strides, dv_strides, scale: Optional[float] = None,
                   delta: Optional[torch.Tensor] = None) -> None:
    """Backward of flash_attn. q/k/v/dq/dk/dv bf16 views with (row, head) strides; o, d_o (B*Nq, H*72) bf16 row-strided;
    lse (B, H, Nq) fp32 from the forward."""
    for t in (q, k, v, o, d_o, dq, dk, dv):
        assert t.dtype == torch.bfloat16 and t.is_cuda
    assert lse.dtype == torch.float32 and lse.is_contiguous() and lse.numel() == B * H * Nq
    assert o.stride(1) == 1 and d_o.stride(1) == 1
    if delta is None:
        delta = torch.empty(B * H * Nq, dtype=torch.float32, device=q.device)
    args = AttnBwdArgs(q=_ptr(q), k=_ptr(k), v=_ptr(v), o=_ptr(o), d_o=_ptr(d_o), lse=_ptr(lse), delta=_ptr(delta),
                       dq=_ptr(dq), dk=_ptr(dk), dv=_ptr(dv), kv_len=_ptr(kv_len), kv_off=_ptr(kv_off),
                       q_sn=q_strides[0], q_sh=q_strides[1], k_sn=k_strides[0], k_sh=k_strides[1],
                       v_sn=v_strides[0], v_sh=v_strides[1], dq_sn=dq_strides[0], dq_sh=dq_strides[1],
                       dk_sn=dk_strides[0], dk_sh=dk_strides[1], dv_sn=dv_strides[0], dv_sh=dv_strides[1],
                       ldo=o.stride(0), lddo=d_o.stride(0), kv_rows=kv_rows, B=B, H=H, Nq=Nq, Nk=Nk,
                       scale=scale if scale is not None else 72 ** -0.5)
    _check(load().pxa_flash_attn_d72_bwd_bf16(C.byref(args), _stream()), "pxa_flash_attn_d72_bwd_bf16")


def gemm_wgrad(a_t: torch.Tensor, w_t: torch.Tensor, out: torch.Tensor, *, block_n: int = 0, k_splits: int = 0,
               max_ctas: int = 0) -> torch.Tensor:
    """out (M, N) fp32 += a_t^T @ w_t with a_t (K, M) and w_t (K, N) bf16 row-major -- the weight gradient
    dW (N_out, K_in) += dY (rows, N_out)^T @ X (rows, K_in) straight from the activations (MN-major UMMA operands, split-K,
    TMA reduce-add into `out`)."""
    assert a_t.dtype == w_t.dtype == torch.bfloat16 and out.dtype == torch.float32
    assert a_t.dim() == 2 and w_t.dim() == 2 and a_t.stride(1) == 1 and w_t.stride(1) == 1 and out.stride(1) == 1
    K, M = a_t.shape
    N = w_t.shape[1]
    assert w_t.shape[0] == K and out.shape == (M, N)
    args = GemmArgs(a=_ptr(a_t), w=_ptr(w_t), bias=None, out=_ptr(out), out_aux_bf16=None, residual=_ptr(out), gate=None,
                    gate_batch_stride=0, rows_per_batch=M, M=M, N=N, K=K, lda=a_t.stride(0), ldw=w_t.stride(0),
                    ldo=out.stride(0), epilogue=EPI_BIAS_RESIDUAL, out_dtype=DTYPE_F32, block_n=block_n, max_ctas=max_ctas,
                    cta_pair=1, debug_trace=None, operands_mn_major=1, k_splits=k_splits, aux_is_branch=0)
    _check(load().pxa_gemm_bf16(C.byref(args), _stream()), "pxa_gemm_bf16 (wgrad)")
    return out


def kv_compress_bwd(k_in, v_in, dk_out, dv_out, dk_in, dv_in, conv_w, conv_b, ln_w, d_conv_w, d_conv_b, d_ln_w, d_ln_b, *,
                    B: int, H: int, W: int, ld_in: int, ld_din: int, eps: float = 1e-5) -> None:
    """Backward of kv_compress: dk_in / dv_in (bf16 views, row stride ld_din) written, the four fp32 parameter gradients
    accumulated."""
    for t in (d_conv_w, d_conv_b, d_ln_w, d_ln_b):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert dk_out.is_contiguous() and dv_out.is_contiguous() and dk_out.dtype == torch.bfloat16
    args = KvCompressBwdArgs(k_in=_ptr(k_in), v_in=_ptr(v_in), dk_out=_ptr(dk_out), dv_out=_ptr(dv_out), dk_in=_ptr(dk_in),
                             dv_in=_ptr(dv_in), conv_w=_ptr(conv_w), conv_b=_ptr(conv_b), ln_w=_ptr(ln_w),
                             d_conv_w=_ptr(d_conv_w), d_conv_b=_ptr(d_conv_b), d_ln_w=_ptr(d_ln_w), d_ln_b=_ptr(d_ln_b),
                             B=B, H=H, W=W, C=dk_out.shape[-1], ld_in=ld_in, ld_din=ld_din, eps=eps)
    _check(load().pxa_kv_compress_conv2_ln_bwd(C.byref(args), _stream()), "pxa_kv_compress_conv2_ln_bwd")
