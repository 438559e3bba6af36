"""Per-tile conditioning cropping == the reference's utils/usdu_utils.py functions on the same inputs.  What
the reference computed is stored in tests/golden/reference_fingerprints.json; the reference_* functions below
recompute it where the reference tree is loadable (oracle/gen_reference_fingerprints.py)."""
import copy

import pytest
import torch

import ref_loader
from __graft_entry__ import load_package
from inputs import fingerprint, reference_fingerprints

load_package()
from comfyui_distributed_b200 import conditioning as C  # noqa: E402

GOLD = reference_fingerprints("test_conditioning")


class FakeControl:
    def __init__(self, hint, prev=None):
        self.cond_hint_original = hint
        self.previous_controlnet = prev

    def copy(self):
        return copy.copy(self)

    def set_previous_controlnet(self, p):
        self.previous_controlnet = p


def _ref():
    ref_loader.load()
    import sys
    return sys.modules[ref_loader.PKG + ".utils.usdu_utils"]


REGIONS = [((480, 992, 1056, 1568), (7680, 4320), (544, 544)), ((0, 0, 544, 544), (1300, 1100), (544, 544)),
           ((724, 524, 1300, 1100), (1300, 1100), (544, 544)), ((10, 20, 170, 150), (300, 260), (160, 136))]


def _key(region, canvas, tile):
    return repr((region, canvas, tile))


def _control(canvas):
    g = torch.Generator().manual_seed(1)
    h1 = torch.rand(1, 3, canvas[1] // 4, canvas[0] // 4, generator=g)
    h2 = torch.rand(2, 3, canvas[1] // 8 + 3, canvas[0] // 8 + 1, generator=g)
    return {"control": FakeControl(h1, FakeControl(h2))}


def _hints(d):
    out, c = [], d["control"]
    while c is not None:
        out.append(c.cond_hint_original)
        c = c.previous_controlnet
    return out


def reference_control_hint_crop(region, canvas, tile):
    d = _control(canvas)
    _ref().crop_controlnet(d, region, canvas, canvas, tile, 0, 0)
    return fingerprint(_hints(d))


@pytest.mark.parametrize("region,canvas,tile", REGIONS)
def test_control_hint_crop_matches_reference(region, canvas, tile):
    mine = _control(canvas)
    C.crop_control_hints(mine, region, canvas, tile)
    hints = _hints(mine)
    assert all(h.shape[-2:] == (tile[1], tile[0]) for h in hints)
    assert fingerprint(hints) == GOLD["control_hint_crop"][_key(region, canvas, tile)]


AREAS = [(40, 60, 10, 20), (8, 8, 0, 0), (500, 500, 3, 7), (1, 1, 400, 400)]
BOXES = [("e1", 20, 30, 5, 6), ("e2", 64, 64, 60, 90), ("e3", 4, 4, 500, 500)]


def _latents(canvas):
    g = torch.Generator().manual_seed(2)
    return [torch.rand(1, 4, canvas[1] // 8, canvas[0] // 8, generator=g), torch.rand(1, 4, 1, 40, 50, generator=g)]


def reference_area_gligen_reflatents(region, canvas, tile):
    u = _ref()
    init = (canvas[0] // 2, canvas[1] // 2)
    areas = []
    for area in AREAS:
        d = {"area": area, "strength": 1.0}
        u.crop_area(d, region, init, canvas, tile, 0, 0)
        areas.append(d)
    gl = {"gligen": ("position", "m", list(BOXES))}
    u.crop_gligen(gl, region, init, canvas, tile, 0, 0)
    lat = {"reference_latents": _latents(canvas)}
    u.crop_reference_latents(lat, region, init, canvas, tile, 0, 0)
    return fingerprint([areas, gl, lat["reference_latents"]])


@pytest.mark.parametrize("region,canvas,tile", REGIONS)
def test_area_gligen_reflatents_match_reference(region, canvas, tile):
    init = (canvas[0] // 2, canvas[1] // 2)
    areas = []
    for area in AREAS:
        d = {"area": area, "strength": 1.0}
        C.crop_area(d, region, init, canvas, 0, 0)
        areas.append(d)
    gl = {"gligen": ("position", "m", list(BOXES))}
    C.crop_gligen(gl, region, init, canvas, 0, 0)
    lat = {"reference_latents": _latents(canvas)}
    C.crop_reference_latents(lat, region, canvas, tile)
    want = GOLD["area_gligen_reflatents"][_key(region, canvas, tile)]
    got = fingerprint([areas, gl, lat["reference_latents"]])
    assert got[0] == want[0] and got[1] == want[1] and got[2] == want[2]


def test_crop_cond_and_clone_do_not_touch_the_originals():
    hint = torch.rand(1, 3, 64, 64)
    cond = [[torch.rand(1, 77, 8), {"control": FakeControl(hint), "area": (8, 8, 0, 0), "pooled_output": torch.rand(1, 8)}]]
    keep = hint.clone()
    out = C.crop_cond(C.clone_conditioning(cond), (0, 0, 128, 128), (256, 256), (256, 256), (128, 128))
    assert torch.equal(hint, keep) and cond[0][1]["control"].cond_hint_original is hint
    assert out[0][1]["control"].cond_hint_original.shape == (1, 3, 128, 128)
    if not torch.cuda.is_available():        # masks are cropped on the GPU only: loud failure, never a CPU path
        from comfyui_distributed_b200._native import NativeError
        with pytest.raises(NativeError):
            C.crop_cond([[None, {"mask": torch.rand(1, 8, 8)}]], (0, 0, 8, 8), (8, 8), (8, 8), (8, 8))
