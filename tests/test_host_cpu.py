"""CPU tests (-m "not gpu"): host-side mirror of the reference interface, C-ABI library surface, build recipe."""
import ctypes
import inspect
import json
import os
import re
import sys
import types

import pytest
import torch

from oracle import pixart_oracle as po
from oracle import refshim
from pixart_sigma_b200 import MODELS, PixArtMS, PixArtMS_XL_2, PixArtMSBlock, build_model, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def reference_surface(golden_dir):
    """What the unmodified reference exposes (tests/golden/reference_surface.json, written by oracle/gen_golden_surface.py)."""
    with open(os.path.join(golden_dir, "reference_surface.json")) as f:
        return json.load(f)


def _tiny(**kw):
    return PixArtMS(depth=2, hidden_size=1152, num_heads=16, input_size=32, pe_interpolation=0.5,
                    model_max_length=300, **kw)


def test_state_dict_layout_matches_reference_checkpoint_keys():
    """Key names AND shapes equal the reference layout restated in the oracle (SURVEY.md 8b)."""
    m = _tiny()
    got = {k: tuple(v.shape) for k, v in m.state_dict().items() if k != "pos_embed"}
    want = po.state_dict_shapes(po.OracleConfig(depth=2))
    assert got == want
    assert tuple(m.state_dict()["pos_embed"].shape) == (1, 256, 1152)


@pytest.mark.parametrize("kw,cfg", [
    (dict(kv_compress_config=dict(sampling="conv", scale_factor=2, kv_compress_layer=[1])),
     dict(kv_sampling="conv", kv_scale_factor=2, kv_compress_layer=[1])),
    (dict(qk_norm=True), dict(qk_norm=True)),
    (dict(micro_condition=True), dict(micro_condition=True)),
])
def test_state_dict_layout_optional_modules(kw, cfg):
    got = {k: tuple(v.shape) for k, v in _tiny(**kw).state_dict().items() if k != "pos_embed"}
    assert got == po.state_dict_shapes(po.OracleConfig(depth=2, **cfg))


def test_state_dict_keys_equal_live_reference(reference_surface):
    ref = {k: tuple(v) for k, v in reference_surface["pixartms_d1_kvconv_state_dict"].items()}
    ours = PixArtMS(depth=1, input_size=32, model_max_length=300,
                    kv_compress_config=dict(sampling="conv", scale_factor=2, kv_compress_layer=[0]))
    os_ = {k: tuple(v.shape) for k, v in ours.state_dict().items()}
    assert os_ == ref
    # a reference checkpoint loads with the same strict=False call the reference scripts use
    sd = {k: torch.randn(v) for k, v in ref.items() if k != "pos_embed"}            # scripts/inference.py:181-184
    missing, unexpected = ours.load_state_dict(sd, strict=False)
    assert missing == ["pos_embed"] and not unexpected


def test_registry_and_builder_surface():
    assert set(MODELS.module_dict) >= {"PixArtMS", "PixArtMS_XL_2"}
    m = build_model(dict(type="PixArtMS", depth=1), use_grad_checkpoint=True, use_fp32_attention=True,
                    input_size=32, model_max_length=300)
    assert isinstance(m, PixArtMS) and m.blocks[0].grad_checkpointing and m.blocks[0].attn.fp32_attention
    assert m.depth == 1 and m.out_channels == 8 and m.patch_size == 2 and m.base_size == 16
    assert isinstance(m.blocks[0], PixArtMSBlock)
    assert callable(PixArtMS_XL_2)


def test_initialisation_zeroes_the_layers_the_reference_zeroes():
    m = _tiny()
    assert float(m.final_layer.linear.weight.abs().sum()) == 0.0
    assert all(float(b.cross_attn.proj.weight.abs().sum()) == 0.0 for b in m.blocks)
    assert float(m.blocks[0].attn.qkv.bias.abs().sum()) == 0.0
    assert 0.015 < float(m.t_block[1].weight.std()) < 0.025


def test_no_cpu_path():
    """The product must fail loudly without the GPU kernels: no eager / CPU fallback exists."""
    m = _tiny().eval()
    x, t, y, _ = po.synthetic_inputs(po.OracleConfig(depth=2), 1, (32, 32))
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU path"):
        m(x, t, y)
    with torch.no_grad(), pytest.raises(RuntimeError, match="no CPU path"):
        m.blocks[0](torch.zeros(1, 256, 1152), torch.zeros(1, 300, 1152), torch.zeros(1, 6 * 1152), [300], (16, 16))


def test_unpatchify_matches_oracle():
    m = _tiny()
    m.h, m.w = 3, 5
    x = torch.randn(2, 15, 32)
    assert torch.equal(m.unpatchify(x), po.unpatchify(x, 3, 5, 2, 8))


def test_library_exports_every_symbol_the_header_declares():
    hdr = open(os.path.join(ROOT, "include", "pixart_sm100.h")).read()
    declared = set(re.findall(r"^\s*(?:int|uint64_t|const char\*)\s+(pxa_\w+)\s*\(", hdr, flags=re.M))
    assert declared == set(lib.EXPORTS)
    dll = lib.load()
    for name in declared:
        assert hasattr(dll, name), name
    assert dll.pxa_version() == 100


def test_ctypes_structs_match_header_sizes():
    """Field-by-field size check of the POD argument structs against a compile of the header with gcc."""
    import subprocess, tempfile
    src = '#include <stdio.h>\n#include "pixart_sm100.h"\nint main(){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(PxaGemmArgs),' \
          ' sizeof(PxaLnModArgs), sizeof(PxaAttnArgs), sizeof(PxaKvCompressArgs), sizeof(PxaConv3x3Args),' \
          ' sizeof(PxaDpmStepArgs), sizeof(PxaGateResidualArgs), sizeof(PxaLnModBwdArgs), sizeof(PxaAttnBwdArgs),' \
          ' sizeof(PxaKvCompressBwdArgs), sizeof(PxaLnPrepareArgs), sizeof(PxaAdamWArgs), sizeof(PxaMlpArgs), sizeof(PxaT5AttnArgs));return 0;}\n'
    with tempfile.TemporaryDirectory() as d:
        open(os.path.join(d, "s.c"), "w").write(src)
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), os.path.join(d, "s.c"), "-o", os.path.join(d, "s")])
        sizes = [int(v) for v in subprocess.check_output([os.path.join(d, "s")]).split()]
    assert sizes == [ctypes.sizeof(lib.GemmArgs), ctypes.sizeof(lib.LnModArgs), ctypes.sizeof(lib.AttnArgs),
                     ctypes.sizeof(lib.KvCompressArgs), ctypes.sizeof(lib.Conv3x3Args), ctypes.sizeof(lib.DpmStepArgs),
                     ctypes.sizeof(lib.GateResidualArgs), ctypes.sizeof(lib.LnModBwdArgs), ctypes.sizeof(lib.AttnBwdArgs),
                     ctypes.sizeof(lib.KvCompressBwdArgs), ctypes.sizeof(lib.LnPrepareArgs), ctypes.sizeof(lib.AdamWArgs), ctypes.sizeof(lib.MlpArgs),
                     ctypes.sizeof(lib.T5AttnArgs)]


def test_integration_md_ctypes_stub_matches_the_header_struct():
    """The binding a reference maintainer would paste from INTEGRATION.md must describe the same PxaAttnArgs as the header
    (a stub that stops short of the trailing pointer fields makes the C side read past the ctypes buffer)."""
    md = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    body = md[md.index("class PxaAttnArgs(C.Structure)"):]
    body = body[:body.index("_lib.pxa_flash_attn_d72_bf16.argtypes")]
    ns = {"C": ctypes}
    exec(body, ns)                                     # noqa: S102 -- our own documentation snippet
    stub = ns["PxaAttnArgs"]
    assert ctypes.sizeof(stub) == ctypes.sizeof(lib.AttnArgs)
    assert [(n, t) for n, t in stub._fields_] == [(n, t) for n, t in lib.AttnArgs._fields_]


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pixart_sigma_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            assert "oracle" not in open(os.path.join(pkg, fn)).read().replace("the oracle", ""), fn


def test_install_into_reference_repoints_registry_and_nets(reference_surface, monkeypatch):
    """INTEGRATION.md level A: after install_into_reference() the reference's own builder / module names construct
    the B200 model, so scripts/inference.py and train_scripts/train.py pick it up unchanged.  The reference package is
    stood in for by modules holding the names it registers and exports (tests/golden/reference_surface.json); its
    `build_model` resolves a model name through `MODELS.build` of the mmcv registry (diffusion/model/builder.py:8-11)."""
    import pixart_sigma_b200
    placeholder = object()
    registry = refshim._Registry("models")
    for name in reference_surface["registry"]:
        registry.register_module(name=name, module=placeholder)
    pkg, model_pkg = types.ModuleType("diffusion"), types.ModuleType("diffusion.model")
    nets, builder = types.ModuleType("diffusion.model.nets"), types.ModuleType("diffusion.model.builder")
    for name in reference_surface["nets"]:
        setattr(nets, name, placeholder)
    builder.MODELS = registry
    pkg.model, model_pkg.nets, model_pkg.builder = model_pkg, nets, builder
    for mod in (pkg, model_pkg, nets, builder):
        monkeypatch.setitem(sys.modules, mod.__name__, mod)
    assert pixart_sigma_b200.install_into_reference()
    assert all(getattr(nets, n) is getattr(pixart_sigma_b200, n) for n in reference_surface["nets"])
    assert all(registry.get(n) is getattr(pixart_sigma_b200, n) for n in reference_surface["registry"])
    m = registry.build(dict(type="PixArtMS"), default_args=dict(depth=1, input_size=32, model_max_length=300))
    assert type(m) is PixArtMS
    # the reference sampler wrapper accepts the model's bound method (diffusion/dpm_solver.py:6-36)
    from diffusion import DPMS
    assert list(inspect.signature(DPMS).parameters) == reference_surface["dpms_params"]
    cond = torch.zeros(1, 1, 300, 4096)
    solver = DPMS(m.forward_with_dpmsolver, condition=cond, uncondition=cond, cfg_scale=4.5,
                  model_kwargs=dict(data_info=None, mask=None))
    assert solver is not None


def test_every_binding_checks_its_return_code_with_one_label():
    """`_check(rc, "name")`: a scripted edit once appended extra labels to one call, which only failed on the GPU box."""
    import ast
    import inspect
    tree = ast.parse(inspect.getsource(lib))
    calls = [n for n in ast.walk(tree) if isinstance(n, ast.Call) and getattr(n.func, "id", None) == "_check"]
    assert len(calls) >= 20 and all(len(n.args) == 2 and not n.keywords for n in calls)


def test_hi_lo_split_of_p_carries_sixteen_mantissa_bits():
    """The arithmetic behind `PxaAttnArgs.p_precision = 1` (DESIGN.md 4.2b): P_hi = bf16(P), P_lo = bf16(P - P_hi) -- the difference is
    exact in fp32 -- so P_hi + P_lo reproduces P to 2^-17 relative (one bf16 term: up to 2^-8), for P anywhere in the lazy-rescale range
    (0, 2^8] incl. values whose low term is subnormal-small."""
    g = torch.Generator().manual_seed(0)
    p = torch.exp2(torch.rand(1 << 16, generator=g) * 40 - 32)                 # 2^-32 .. 2^8
    hi = p.to(torch.bfloat16)
    diff = p - hi.float()
    assert torch.equal(diff.double(), p.double() - hi.double())               # exact in fp32
    lo = diff.to(torch.bfloat16)
    err1 = ((hi.double() - p.double()).abs() / p.double()).max().item()
    err2 = ((hi.double() + lo.double() - p.double()).abs() / p.double()).max().item()
    assert 2.0 ** -9 < err1 <= 2.0 ** -8 and err2 <= 2.0 ** -17


def test_single_scale_pixart_surface_equals_live_reference(reference_surface):
    """nets/PixArt.py: `PixArt` / `PixArt_XL_2` / `PixArtBlock` (the 256px Sigma config builds `PixArt_XL_2`,
    configs/pixart_sigma_config/PixArt_sigma_xl2_img256_internal.py:12): same state-dict keys and shapes as the unmodified reference
    class, registry names, the single-scale forward signatures (tests/golden/reference_surface.json)."""
    from pixart_sigma_b200 import PixArt, PixArt_XL_2, PixArtBlock
    kv = dict(sampling="conv", scale_factor=2, kv_compress_layer=[1])
    ours = PixArt(input_size=16, depth=2, model_max_length=300, qk_norm=True, kv_compress_config=kv)
    ref = {k: tuple(v) for k, v in reference_surface["pixart_single_scale_state_dict"].items()}
    assert {k: tuple(v.shape) for k, v in ours.state_dict().items()} == ref
    ours.load_state_dict({k: torch.randn(v) for k, v in ref.items()}, strict=True)
    assert set(MODELS.module_dict) >= set(reference_surface["registry"])
    assert isinstance(build_model("PixArt", depth=1, input_size=8), PixArt) and callable(PixArt_XL_2)
    assert all(type(b) is PixArtBlock for b in ours.blocks) and not ours.micro_conditioning and ours.out_channels == 8
    for name in ("forward", "forward_with_dpmsolver", "forward_with_cfg"):
        ours_p = list(inspect.signature(getattr(PixArt, name)).parameters)
        ref_p = reference_surface["pixart_signatures"][name]
        assert ours_p == ref_p, (name, ours_p, ref_p)
    assert list(inspect.signature(PixArtBlock.forward).parameters)[:5] == ["self", "x", "y", "t", "mask"]
    with pytest.raises(ValueError, match="single-scale"):
        ours(torch.zeros(1, 4, 32, 32), torch.zeros(1), torch.zeros(1, 1, 300, 4096))
    with pytest.raises(RuntimeError):                      # right size: reaches the kernel path, which refuses CPU tensors
        ours(torch.zeros(1, 4, 16, 16), torch.zeros(1), torch.zeros(1, 1, 300, 4096))
