"""TEST INFRASTRUCTURE ONLY -- run the key-mapping body of the UNMODIFIED reference converter
(`tools/convert_pixart_to_diffusers.py:27-154` of the reference checkout that oracle/refshim.py finds, exec'd on a synthetic
small-width state dict with the reference key layout) and store what it produced: tests/golden/diffusers_mapping.pt =
{diffusers key: (shape, sum, sum of magnitudes)} plus a position-weighted sum per key (`weighted_sum`, which a reordering inside
a tensor changes) for the plain, micro-condition and qk-norm variants.  Needs the reference checkout."""
import os
import sys
import textwrap
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import pixart_oracle as po  # noqa: E402
from oracle.refshim import REFERENCE_ROOT  # noqa: E402

REF = os.path.join(REFERENCE_ROOT, "tools", "convert_pixart_to_diffusers.py")


def weighted_sum(v: torch.Tensor) -> float:
    """sum_i cos(i) * v.flatten()[i] in float64: unlike the plain sums it changes when elements swap places."""
    flat = v.detach().double().flatten()
    return float((flat * torch.arange(flat.numel(), dtype=torch.float64).cos()).sum())


def small_state_dict(micro: bool, qk: bool):
    cfg = po.OracleConfig(depth=28, hidden_size=32, num_heads=2, micro_condition=micro, qk_norm=qk)
    return po.synthetic_state_dict(cfg, seed=3)


def reference_mapping(sd, micro: bool, qk: bool):
    src = open(REF).read().splitlines()
    start = next(i for i, l in enumerate(src) if "converted_state_dict = {}" in l)
    end = next(i for i, l in enumerate(src) if "# PixArt XL/2" in l)
    ns = {"torch": torch, "state_dict": dict(sd),
          "args": SimpleNamespace(micro_condition=micro, qk_norm=qk, version="alpha", image_size=1024)}
    exec(textwrap.dedent("\n".join(src[start:end])), ns)
    return ns["converted_state_dict"], ns["state_dict"]


def main():
    fix = {}
    for name, micro, qk in (("plain", False, False), ("micro", True, False), ("qknorm", False, True)):
        sd = small_state_dict(micro, qk)
        conv, left = reference_mapping(sd, micro, qk)
        fix[name] = {"micro": micro, "qk": qk, "left_over": sorted(left),
                     "entries": {k: (tuple(v.shape), float(v.double().sum()), float(v.double().abs().sum())) for k, v in conv.items()},
                     "weighted_sum": {k: weighted_sum(v) for k, v in conv.items()}}
        print(name, len(conv), "converted keys,", len(left), "left over:", sorted(left))
    torch.save(fix, os.path.join(ROOT, "tests", "golden", "diffusers_mapping.pt"))


if __name__ == "__main__":
    main()
