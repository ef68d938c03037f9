"""TEST INFRASTRUCTURE ONLY -- dependency stand-ins that let the *unmodified* reference
(`/root/reference`, PixArt-alpha/PixArt-sigma) import in this container.

The reference needs timm==0.6.12, xformers==0.0.19 and mmcv==1.7.0 (requirements.txt:1-19), none of
which are installed and there is no network.  This module injects minimal `sys.modules` stand-ins
that restate the *published* behaviour of the few symbols the hot path touches:

  timm.models.vision_transformer.{Mlp, Attention, PatchEmbed}, timm.models.layers.DropPath
      (call sites: diffusion/model/nets/PixArtMS.py:13-14,67; PixArt_blocks.py:17,61,385; PixArt.py:16-17)
  xformers.ops.memory_efficient_attention, xformers.ops.fmha.BlockDiagonalMask.from_seqlens
      (call sites: PixArt_blocks.py:52-53,153) -- softmax(q k^T * K^-0.5) v in fp32 math via SDPA
  mmcv.Registry / mmcv.runner.get_dist_info / mmcv.utils.logging.logger_initialized
      (call sites: diffusion/model/builder.py:1,5,11; diffusion/utils/logger.py:6; dist_utils.py:10,13)

Nothing here is imported by the product package `pixart_sigma_b200`; it is used by the
`oracle/gen_golden*.py` fixture generators, which need a reference checkout, and the registry stand-in
by `tests/test_host_cpu.py`, which needs none.
"""
import os
import sys
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

REFERENCE_ROOT = os.environ.get("PIXART_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "diffusion", "model", "nets"))


# ----------------------------------------------------------------------------- timm
class _DropPath(nn.Module):
    def __init__(self, drop_prob=0.0, scale_by_keep=True):
        super().__init__()
        self.drop_prob = drop_prob

    def forward(self, x):
        if self.drop_prob == 0.0 or not self.training:
            return x
        keep = 1.0 - self.drop_prob
        m = x.new_empty((x.shape[0],) + (1,) * (x.ndim - 1)).bernoulli_(keep)
        return x * m / keep


class _Mlp(nn.Module):
    """timm 0.6.12 Mlp: fc1 -> act -> drop1 -> fc2 -> drop2 (act_layer is *instantiated*)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU,
                 bias=True, drop=0.0):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias)
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop)
        self.fc2 = nn.Linear(hidden_features, out_features, bias=bias)
        self.drop2 = nn.Dropout(drop)

    def forward(self, x):
        return self.drop2(self.fc2(self.drop1(self.act(self.fc1(x)))))


class _Attention(nn.Module):
    """timm 0.6.12 Attention ctor surface (forward is overridden by the reference)."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, attn_drop=0.0, proj_drop=0.0, **_):
        super().__init__()
        assert dim % num_heads == 0
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)


class _TimmPatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768, norm_layer=None,
                 flatten=True, bias=True):
        super().__init__()
        img_size = (img_size, img_size) if isinstance(img_size, int) else tuple(img_size)
        patch_size = (patch_size, patch_size) if isinstance(patch_size, int) else tuple(patch_size)
        self.img_size, self.patch_size = img_size, patch_size
        self.grid_size = (img_size[0] // patch_size[0], img_size[1] // patch_size[1])
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.flatten = flatten
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size, bias=bias)
        self.norm = norm_layer(embed_dim) if norm_layer else nn.Identity()

    def forward(self, x):
        x = self.proj(x)
        if self.flatten:
            x = x.flatten(2).transpose(1, 2)
        return self.norm(x)


# ----------------------------------------------------------------------------- xformers
class _BlockDiagonalMask:
    def __init__(self, q_seqlen, kv_seqlen):
        self.q_seqlen, self.kv_seqlen = list(q_seqlen), list(kv_seqlen)

    @classmethod
    def from_seqlens(cls, q_seqlen, kv_seqlen=None):
        return cls(q_seqlen, q_seqlen if kv_seqlen is None else kv_seqlen)


def _sdpa(q, k, v, attn_mask=None, scale=None):
    # xformers layout (B, M, H, K) -> SDPA layout (B, H, M, K); default scale K^-0.5
    o = F.scaled_dot_product_attention(q.transpose(1, 2), k.transpose(1, 2), v.transpose(1, 2),
                                       attn_mask=attn_mask, scale=scale)
    return o.transpose(1, 2)


def _memory_efficient_attention(query, key, value, attn_bias=None, p=0.0, scale=None, **_):
    if isinstance(attn_bias, _BlockDiagonalMask):
        outs, qo, ko = [], 0, 0
        for ql, kl in zip(attn_bias.q_seqlen, attn_bias.kv_seqlen):
            ql, kl = int(ql), int(kl)
            if kl == 0:  # empty key set: xformers yields zeros for these queries
                outs.append(torch.zeros_like(query[:, qo:qo + ql]))
            else:
                outs.append(_sdpa(query[:, qo:qo + ql], key[:, ko:ko + kl], value[:, ko:ko + kl], scale=scale))
            qo += ql
            ko += kl
        return torch.cat(outs, dim=1)
    mask = None
    if attn_bias is not None:  # dense additive bias (B*H, M, N)
        B, M, H, _ = query.shape
        mask = attn_bias.reshape(B, H, M, -1)
    return _sdpa(query, key, value, attn_mask=mask, scale=scale)


# ----------------------------------------------------------------------------- mmcv
class _Registry:
    def __init__(self, name):
        self.name, self._m = name, {}

    def register_module(self, name=None, force=False, module=None):
        def deco(obj):
            self._m[name or obj.__name__] = obj
            return obj
        return deco(module) if module is not None else deco

    def get(self, key):
        return self._m.get(key)

    @property
    def module_dict(self):
        return self._m

    def build(self, cfg, default_args=None):
        args = dict(cfg)
        if default_args:
            for k, v in default_args.items():
                args.setdefault(k, v)
        typ = args.pop("type")
        fn = self._m[typ] if isinstance(typ, str) else typ
        return fn(**args)


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_reference_shims(force: bool = False) -> None:
    """Inject the stand-ins (only for packages that are genuinely missing) and put the reference on sys.path."""
    def missing(pkg):
        if force:
            return True
        if pkg in sys.modules:
            return False
        import importlib.util
        return importlib.util.find_spec(pkg) is None

    if missing("timm"):
        timm = _mod("timm"); models = _mod("timm.models")
        layers = _mod("timm.models.layers", DropPath=_DropPath)
        vt = _mod("timm.models.vision_transformer", Mlp=_Mlp, Attention=_Attention, PatchEmbed=_TimmPatchEmbed)
        timm.models, models.layers, models.vision_transformer = models, layers, vt
    if missing("xformers"):
        xf = _mod("xformers")
        fmha = _mod("xformers.ops.fmha", BlockDiagonalMask=_BlockDiagonalMask)
        ops = _mod("xformers.ops", memory_efficient_attention=_memory_efficient_attention, fmha=fmha)
        xf.ops = ops
    if missing("mmcv"):
        mmcv = _mod("mmcv", Registry=_Registry)
        runner = _mod("mmcv.runner", get_dist_info=lambda: (0, 1))
        utils = _mod("mmcv.utils")
        logging_ = _mod("mmcv.utils.logging", logger_initialized={})
        mmcv.runner, mmcv.utils, utils.logging = runner, utils, logging_
    if reference_available() and REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)


def load_reference_model(**kwargs):
    """Build the reference's own PixArtMS_XL_2 (fp32, CPU) through the shims."""
    install_reference_shims()
    from diffusion.model.nets.PixArtMS import PixArtMS_XL_2  # noqa: the reference, unmodified
    return PixArtMS_XL_2(**kwargs)
