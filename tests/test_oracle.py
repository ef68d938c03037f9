"""CPU tests (-m "not gpu"): the oracle restatement against the committed golden fixtures that
oracle/gen_golden.py and oracle/gen_golden_surface.py produced from the UNMODIFIED reference."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import pixart_oracle as po
from oracle.gen_golden_surface import ragged_inputs

TOL = 2e-5  # fp32 vs fp32, different op order only


def _run_case(fix):
    cfg = po.OracleConfig(**fix["cfg"])
    sd = po.synthetic_state_dict(cfg, seed=0)
    x, t, y, mask = po.synthetic_inputs(cfg, fix["batch"], tuple(fix["hw"]), seed=0, timesteps=fix["t"], lens=fix["lens"])
    data_info = None
    if fix["micro"]:
        data_info = {"img_hw": torch.tensor([[256.0, 256.0]]).repeat(fix["batch"], 1),
                     "aspect_ratio": torch.tensor([[1.0]]).repeat(fix["batch"], 1)}
    return po.forward(sd, cfg, x, t, y, mask=mask, data_info=data_info, return_intermediates=True)


def _cases(golden_dir, depth28):
    out = []
    for p in sorted(glob.glob(os.path.join(golden_dir, "*.pt"))):
        name = os.path.basename(p)[:-3]
        if name.startswith("xl2_") == depth28:
            out.append(p)
    return out


def test_golden_fixtures_exist(golden_dir):
    assert len(glob.glob(os.path.join(golden_dir, "d2_*.pt"))) >= 8
    assert len(glob.glob(os.path.join(golden_dir, "xl2_*.pt"))) >= 1


@pytest.mark.parametrize("name", ["d2_nomask", "d2_nonsquare", "d2_kvconv", "d2_kvave", "d2_kvuniform",
                                  "d2_kvuniform_every", "d2_qknorm", "d2_micro", "d2_emptykeys"])
def test_oracle_matches_reference_golden_depth2(golden_dir, name):
    fix = torch.load(os.path.join(golden_dir, name + ".pt"))
    out, inter = _run_case(fix)
    assert out.shape == fix["out"].shape
    assert po.rel_err(out, fix["out"]) < TOL
    assert po.rel_err(inter["blocks"][0][:, ::37], fix["block0_tap"]) < TOL
    assert po.rel_err(inter["blocks"][-1][:, ::37], fix["block_last_tap"]) < TOL


@pytest.mark.slow
@pytest.mark.parametrize("name", ["xl2_256_b1_mask77"])
def test_oracle_matches_reference_golden_xl2(golden_dir, name):
    """BASELINE config c1: PixArt-Sigma-XL/2 256px single forward on CPU (the correctness gate)."""
    fix = torch.load(os.path.join(golden_dir, name + ".pt"))
    out, inter = _run_case(fix)
    assert po.rel_err(out, fix["out"]) < 5e-5
    assert po.rel_err(inter["blocks"][-1][:, ::37], fix["block_last_tap"]) < 5e-5


def test_pos_embed_against_reference_formula():
    """sincos table: first half of channels encodes the w axis, [sin|cos] per quarter (PixArt.py:258-307)."""
    e = po.sincos_pos_embed(1152, 3, 5, pe_interpolation=2.0, base_size=64)
    assert e.shape == (15, 1152) and e.dtype == np.float64
    pos_w = np.arange(5, dtype=np.float32) / (5 / 64) / 2.0
    pos_h = np.arange(3, dtype=np.float32) / (3 / 64) / 2.0
    om = 1.0 / 10000 ** (np.arange(288, dtype=np.float64) / 288)
    tok = 1 * 5 + 3                                   # (row 1, col 3)
    np.testing.assert_allclose(e[tok, 0:288], np.sin(pos_w[3] * om), rtol=0, atol=1e-12)
    np.testing.assert_allclose(e[tok, 288:576], np.cos(pos_w[3] * om), rtol=0, atol=1e-12)
    np.testing.assert_allclose(e[tok, 576:864], np.sin(pos_h[1] * om), rtol=0, atol=1e-12)


def test_state_dict_layout_matches_survey_counts():
    """437 tensors / 610,856,096 params for XL/2 (+y_embedding, -pos_embed buffers); SURVEY.md Appendix A."""
    cfg = po.OracleConfig(depth=28, model_max_length=300)
    shapes = po.state_dict_shapes(cfg)
    # reference state_dict has 437 entries incl. the pos_embed buffer, which is dropped on load
    assert len(shapes) == 436
    n_params = sum(int(np.prod(s)) for k, s in shapes.items() if k != "y_embedder.y_embedding")
    assert n_params == 610_856_096
    kv = po.OracleConfig(depth=28, kv_sampling="conv", kv_scale_factor=2, kv_compress_layer=list(range(14, 28)))
    assert len(po.state_dict_shapes(kv)) == 492


def test_oracle_matches_live_reference_ragged_mask(golden_dir):
    """Against the unmodified reference with a NON-prefix 0/1 mask (masked_select semantics); its outputs are stored in
    tests/golden/ragged_mask_d1.pt (oracle/gen_golden_surface.py)."""
    fix = torch.load(os.path.join(golden_dir, "ragged_mask_d1.pt"))
    cfg, sd, x, t, y, mask = ragged_inputs()
    got = po.forward(sd, cfg, x, t, y, mask=mask)
    assert po.rel_err(got, fix["out"]) < TOL
    # batch-broadcast 2-D mask (CFG: n masks for 2n samples, PixArtMS.py:197-198) ...
    got2 = po.forward(sd, cfg, x, t, y, mask=mask[:1])
    assert po.rel_err(got2, fix["out_mask_broadcast"]) < TOL
    # ... and the trainer's (B,1,1,L) layout (train.py:158-168; squeezed at PixArtMS.py:199)
    got3 = po.forward(sd, cfg, x, t, y, mask=mask.reshape(2, 1, 1, 300))
    assert po.rel_err(got3, fix["out_mask_b11l"]) < TOL
