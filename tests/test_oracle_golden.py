"""Pin the oracle against fixtures produced by RUNNING the real reference
(oracle/gen_golden.py; reference @ a91f9fb).  Bit-exact."""
import hashlib
import json
import os

import numpy as np
import pytest

import usdu_oracle as orc
from inputs import make_input

G = os.path.join(os.path.dirname(__file__), "golden")
GEO = json.load(open(os.path.join(G, "geometry.json")))["cases"]
SINGLE = json.load(open(os.path.join(G, "single_index.json")))["cases"]


@pytest.mark.parametrize("case", GEO, ids=lambda c: f"{c['W']}x{c['H']}_t{c['tile_w']}x{c['tile_h']}_p{c['padding']}_{'u' if c['uniform'] else 'n'}")
def test_geometry_matches_reference(case):
    tw, th, plan = orc.make_plan(case["W"], case["H"], case["tile_w"], case["tile_h"], case["padding"], case["uniform"])
    assert (tw, th) == (case["tw"], case["th"])
    rows = [[t.x, t.y, t.x1, t.y1, t.ew, t.eh, t.pw, t.ph] for t in plan]
    assert rows == case["rows"]


def test_mask_and_blend_match_reference():
    p = np.load(os.path.join(G, "prims.npz"))
    rng = np.random.default_rng(1234)               # the inputs oracle/gen_golden.py gave the reference's blend_tile
    for i in range(4):
        W, H, x, y, tw, th, blur, pad, x1, y1, x2, y2, pw, ph = [int(v) for v in p[f"case{i}_params"]]
        m = orc.tile_mask_window(W, H, x, y, tw, th, blur, (x1, y1, x2, y2))
        assert np.array_equal(m, p[f"case{i}_mask"][y1:y2, x1:x2])
        base = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        tile = rng.integers(0, 256, (ph, pw, 3), dtype=np.uint8)
        want = base.copy()                          # the reference left every pixel outside the window as it was
        want[y1:y2, x1:x2] = p[f"case{i}_out_window"]
        r = orc.lanczos_resize_u8(tile, x2 - x1, y2 - y1) if (pw, ph) != (x2 - x1, y2 - y1) else tile
        base[y1:y2, x1:x2] = orc.composite_u8(r, base[y1:y2, x1:x2], m)
        assert np.array_equal(base, want)


@pytest.mark.parametrize("case", SINGLE, ids=lambda c: c["name"])
def test_process_single_matches_reference(case):
    img = make_input(case["kind"], case["seed"], case["B"], case["H"], case["W"])
    res = orc.process_single(img, orc.make_t0_denoiser(case["denoise_seed"], case["denoise"]), case["tile_w"],
                             case["tile_h"], case["padding"], case["mask_blur"], case["uniform"])
    out = orc.quantize_u8(res)
    assert np.array_equal(orc.dequantize_u8(out), res)
    ref = np.load(os.path.join(G, f"single_{case['name']}.npz"))["out"]
    assert hashlib.sha256(ref.tobytes()).hexdigest() == case["sha256"]
    assert np.array_equal(out, ref)


def test_mask_crop_matches_reference():
    """oracle.crop_mask_u8 == the reference's crop_mask (utils/usdu_utils.py:415-442), fixtures from
    oracle/gen_golden.py."""
    from inputs import MASK_CROP_CASES, make_mask
    gold = np.load(os.path.join(G, "mask_crop.npz"))
    for (name, kind, seed, B, (Hm, Wm), region, canvas, tile) in MASK_CROP_CASES:
        m = make_mask(kind, seed, B, Hm, Wm)
        for b in range(B):
            got = orc.crop_mask_u8(orc.quantize_u8(m[b]), region, canvas, tile)
            assert np.array_equal(got, gold[name][b]), name


STATIC_REF = json.load(open(os.path.join(G, "static_ref_index.json")))["cases"]


@pytest.mark.parametrize("case", STATIC_REF, ids=lambda c: c["name"])
def test_replay_static_matches_the_reference_run_over_http(case):
    """oracle.replay_static with the RECORDED tile assignment == what the reference's own static mode
    (master + workers, aiohttp + PNG transport, really run by oracle/ref_static_run.py) produced."""
    img = make_input(case["kind"], case["seed"], case["B"], case["H"], case["W"])
    res = orc.replay_static(img, orc.make_t0_denoiser(case["denoise_seed"], case["denoise"]), case["tile"], case["tile"],
                            case["padding"], case["mask_blur"], case["uniform"], case["assignment"])
    assert hashlib.sha256(orc.quantize_u8(res).tobytes()).hexdigest() == case["sha256"]


SWEEP_DIGESTS = json.load(open(os.path.join(G, "sweep_ref_digests.json")))["digests"]


def _sweep_subset():
    from inputs import sweep_cases
    cs = sweep_cases()
    return cs[::3] + cs[-4:]          # every third case + the four hand-picked extremes (all 44 run on the GPU box)


@pytest.mark.parametrize("case", _sweep_subset(), ids=lambda c: f"{c[0]}-{c[1]}-b{c[2]}-{c[4]}x{c[3]}")
def test_oracle_matches_reference_digests_of_the_parameter_sweep(case):
    from inputs import sweep_sampler
    i, kind, B, H, W, tw, th, pad, blur, uniform = case
    seed, den = sweep_sampler(i)
    res = orc.process_single(make_input(kind, i, B, H, W), orc.make_t0_denoiser(seed, den), tw, th, pad, blur, uniform)
    assert hashlib.sha256(orc.quantize_u8(res).tobytes()).hexdigest() == SWEEP_DIGESTS[str(i)]
