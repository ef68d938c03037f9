"""TEST INFRASTRUCTURE ONLY -- record what the CPU tests compare against from the UNMODIFIED reference (imported through
oracle/refshim.py; point PIXART_REFERENCE_ROOT at a checkout of PixArt-alpha/PixArt-sigma), so that the tests run without it:

  tests/golden/reference_surface.json  state-dict keys and shapes of two small reference models, the forward signatures of the
                                       single-scale `PixArt`, the names the reference registers in `diffusion.model.builder.MODELS`
                                       and exports from `diffusion.model.nets`, and the parameters of `diffusion.DPMS`
  tests/golden/ragged_mask_d1.pt       one-block `PixArtMS` outputs for a NON-prefix 0/1 caption mask in the three layouts the
                                       reference accepts (per sample, batch-broadcast, the trainer's (B, 1, 1, L))

Weights and inputs are regenerated from seeds by `oracle.pixart_oracle`; only the reference's results are stored.
    python oracle/gen_golden_surface.py
"""
import inspect
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pixart_oracle as po                      # noqa: E402
from oracle.refshim import install_reference_shims, reference_available  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")

# the models whose state-dict layout the tests pin (tests/test_host_cpu.py)
MS_CFG = po.OracleConfig(depth=1, kv_sampling="conv", kv_scale_factor=2, kv_compress_layer=[0])
SINGLE_SCALE_KW = dict(input_size=16, depth=2, model_max_length=300, qk_norm=True,
                       kv_compress_config=dict(sampling="conv", scale_factor=2, kv_compress_layer=[1]))

# the ragged-mask case (tests/test_oracle.py)
RAGGED_CFG = dict(depth=1, input_size=32, pe_interpolation=0.5)
RAGGED_SEED, RAGGED_HW, RAGGED_T, RAGGED_MASK_SEED = 3, (16, 24), [749.25, 3.0], 5


def ragged_inputs():
    cfg = po.OracleConfig(**RAGGED_CFG)
    sd = po.synthetic_state_dict(cfg, seed=RAGGED_SEED)
    x, t, y, _ = po.synthetic_inputs(cfg, 2, RAGGED_HW, seed=RAGGED_SEED, timesteps=RAGGED_T)
    mask = (torch.rand(2, 300, generator=torch.Generator().manual_seed(RAGGED_MASK_SEED)) > 0.5).long()
    return cfg, sd, x, t, y, mask


def _shapes(module):
    return {k: list(v.shape) for k, v in module.state_dict().items()}


def surface():
    from diffusion import DPMS
    from diffusion.model import nets
    from diffusion.model.builder import MODELS
    from diffusion.model.nets.PixArt import PixArt
    from oracle.gen_golden import build_reference
    return {
        "pixartms_d1_kvconv_state_dict": _shapes(build_reference(MS_CFG, po.synthetic_state_dict(MS_CFG))),
        "pixart_single_scale_state_dict": _shapes(PixArt(**SINGLE_SCALE_KW)),
        "pixart_signatures": {n: list(inspect.signature(getattr(PixArt, n)).parameters)
                              for n in ("forward", "forward_with_dpmsolver", "forward_with_cfg")},
        "registry": sorted(MODELS.module_dict),
        "nets": sorted(n for n, v in vars(nets).items() if n.startswith("PixArt") and not inspect.ismodule(v)),
        "dpms_params": list(inspect.signature(DPMS).parameters),
    }


def ragged_outputs():
    from oracle.gen_golden import build_reference
    cfg, sd, x, t, y, mask = ragged_inputs()
    ref = build_reference(cfg, sd)
    with torch.no_grad():
        return {"out": ref(x, t, y, mask=mask, data_info=None),
                "out_mask_broadcast": ref(x, t, y, mask=mask[:1], data_info=None),
                "out_mask_b11l": ref(x, t, y, mask=mask.reshape(2, 1, 1, 300), data_info=None)}


def main():
    assert reference_available(), "set PIXART_REFERENCE_ROOT to a checkout of the reference"
    install_reference_shims()
    with open(os.path.join(OUT, "reference_surface.json"), "w") as f:
        json.dump(surface(), f, indent=1, sort_keys=True)
        f.write("\n")
    torch.save(ragged_outputs(), os.path.join(OUT, "ragged_mask_d1.pt"))


if __name__ == "__main__":
    main()
