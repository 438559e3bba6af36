"""denoise.ComfySampler (our per-tile VAEEncode -> common_ksampler -> VAEDecode driver) next to the
reference's own process_tiles_batch (upscale/tile_ops.py:239-287), both against the same recording
stand-in for ComfyUI's `nodes` module: the sampler must be called with the same pixels, seed/steps/cfg/...,
the same cropped ControlNet hints / areas / GLIGEN boxes, the same tile-local model patch, in the same
order, and hand back the same pixels.  CPU only.  What the reference's side saw and returned is stored in
tests/golden/reference_fingerprints.json; reference_process_tiles_batch recomputes it where the reference tree is
loadable (oracle/gen_reference_fingerprints.py)."""
import copy
import sys
import types

import pytest
import torch

import ref_loader
from __graft_entry__ import load_package
from inputs import fingerprint, reference_fingerprints

load_package()
from comfyui_distributed_b200 import planner  # noqa: E402
from comfyui_distributed_b200.conditioning import make_cond_cropper  # noqa: E402
from comfyui_distributed_b200.denoise import ComfySampler  # noqa: E402

class FakeControl:
    def __init__(self, hint, prev=None):
        self.cond_hint_original = hint
        self.previous_controlnet = prev

    def copy(self):
        return copy.copy(self)

    def set_previous_controlnet(self, p):
        self.previous_controlnet = p


class DiffSynthCnetPatch:
    def __init__(self, model_patch, vae, image, strength, inpaint_image=None, mask=None):
        self.model_patch, self.vae, self.image, self.strength = model_patch, vae, image, strength
        self.inpaint_image, self.mask = inpaint_image, mask
        self.encoded_image, self.encoded_image_size = None, (image.shape[1], image.shape[2])


class Model:
    def __init__(self, patch):
        self.patch = patch
        self.model_options = {"transformer_options": {"patches": {"double_block": [patch]}}}

    def clone(self):
        return Model(self.patch)


def _recording_nodes(log, tiled=()):
    class VAEEncode:
        def encode(self, vae, px):
            log.append(("encode", px.clone()))
            return ({"samples": px * 0.5},)

    class VAEDecode:
        def decode(self, vae, s):
            log.append(("decode", s["samples"].clone()))
            return (s["samples"] + 0.25,)

    def common_ksampler(model, seed, steps, cfg, sampler_name, scheduler, pos, neg, latent, denoise=1.0):
        def view(cond):
            out = []
            for emb, d in cond:
                c, hints = d.get("control"), []
                while c is not None:
                    hints.append(c.cond_hint_original.clone())
                    c = c.previous_controlnet
                gl = d.get("gligen")
                out.append((emb.clone(), hints, d.get("area"), d.get("strength"), None if gl is None else [b[1:] for b in gl[2]]))
            return out
        log.append(("sample", seed, steps, cfg, sampler_name, scheduler, denoise, view(pos), view(neg),
                    latent["samples"].clone(), model.patch.image.clone(), tuple(model.patch.encoded_image_size)))
        return ({"samples": latent["samples"] * 2.0},)

    class VAEDecodeTiled:
        def decode(self, vae, s, tile_size=None):
            log.append(("decode_tiled", s["samples"].clone(), tile_size))
            return (s["samples"] + 0.5,)

    ns = types.SimpleNamespace(VAEEncode=VAEEncode, VAEDecode=VAEDecode, common_ksampler=common_ksampler)
    if "decode" in tiled:
        ns.VAEDecodeTiled = VAEDecodeTiled
    if "encode" in tiled:
        ns.VAEEncodeTiled = object
    return ns


CASES = [(700, 520, 256, 32, True), (420, 300, 128, 16, False)]
TILED = [(False, ()), (True, ("encode", "decode")), (True, ("decode",)), (True, ())]


def _side(side, W, H, tile, pad, uniform, tiled_decode, tiled):
    """Every tile of the plan through one side ("ref": the reference's process_tiles_batch, "new": ComfySampler)
    -> [(tile index, returned pixels, calls the recording `nodes` saw)]."""
    g = torch.Generator().manual_seed(1)
    B = 2
    hint = torch.rand(1, 3, H // 2, W // 2, generator=g)
    hint2 = torch.rand(1, 3, H // 4, W // 4, generator=g)
    control_image = torch.rand(1, H // 2, W // 2, 3, generator=g)
    gligen = ("position", "gligen-model", [(torch.rand(1, 8, generator=g), 8, 10, 4, 6), (torch.rand(1, 8, generator=g), 20, 12, 30, 40)])

    def make_cond():
        return [[torch.rand(1, 77, 8, generator=torch.Generator().manual_seed(2)),
                 {"control": FakeControl(hint, FakeControl(hint2)), "area": (16, 24, 8, 4), "strength": 0.7, "gligen": gligen,
                  "pooled_output": torch.zeros(1, 8)}]]

    p = planner.Plan.build(W, H, tile, tile, pad, 8, uniform)
    args = (123, 7, 4.5, "euler", "normal", 0.35)
    tile_ops = ref_loader.load()[0] if side == "ref" else None
    res = []
    for t in p.tiles:
        px = torch.rand(B, t.ph, t.pw, 3, generator=g)
        log = []
        saved = sys.modules.get("nodes")
        sys.modules["nodes"] = _recording_nodes(log, tiled)
        try:
            model = Model(DiffSynthCnetPatch("mp", None, control_image.clone(), 1.0))
            pos, neg = make_cond(), make_cond()
            if side == "ref":
                out = tile_ops.TileOpsMixin().process_tiles_batch(px.clone(), model, pos, neg, "vae", *args, tiled_decode,
                                                                  (t.x1, t.y1, t.x2, t.y2), (W, H))
            else:
                s = ComfySampler(model, pos, neg, "vae", *args, tiled_decode=tiled_decode, image_size=(W, H),
                                 cond_cropper=make_cond_cropper())
                out = s(px.clone()[None], [t])[0]
        finally:
            if saved is None:
                sys.modules.pop("nodes", None)
            else:
                sys.modules["nodes"] = saved
        assert torch.equal(model.patch.image, control_image)          # patch restored after the tile
        res.append((t.idx, out, log))
    return res


def _key(W, H, tile, pad, uniform, tiled_decode, tiled):
    return repr((W, H, tile, pad, uniform, tiled_decode, tiled))


def reference_process_tiles_batch(W, H, tile, pad, uniform, tiled_decode, tiled):
    return [{"idx": i, "out": fingerprint(out), "log": [fingerprint(c) for c in log]}
            for i, out, log in _side("ref", W, H, tile, pad, uniform, tiled_decode, tiled)]


@pytest.mark.parametrize("tiled_decode,tiled", TILED)
@pytest.mark.parametrize("W,H,tile,pad,uniform", CASES)
def test_sampler_driver_matches_process_tiles_batch(W, H, tile, pad, uniform, tiled_decode, tiled):
    want = reference_fingerprints("test_comfy_sampler_vs_reference")["process_tiles_batch"][
        _key(W, H, tile, pad, uniform, tiled_decode, tiled)]
    got = _side("new", W, H, tile, pad, uniform, tiled_decode, tiled)
    assert len(got) == len(want)
    for (idx, out, log), w in zip(got, want):
        assert idx == w["idx"]
        assert fingerprint(out) == w["out"], idx
        assert len(log) == len(w["log"]) == 3
        for call, wc in zip(log, w["log"]):
            assert fingerprint(call) == wc, (idx, call[0])
