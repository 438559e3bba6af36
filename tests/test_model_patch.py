"""Tile-local model patches == the reference's crop_model_cond (utils/crop_model_patch.py) on the same fake
ComfyUI objects (what the reference computed: tests/golden/reference_fingerprints.json, recomputed by
reference_crop_model_cond where the reference tree is loadable), plus behaviour checks."""
import sys

import pytest
import torch

import ref_loader
from __graft_entry__ import load_package
from inputs import fingerprint, reference_fingerprints

load_package()
from comfyui_distributed_b200 import model_patch as MP  # noqa: E402


class FakeVAE:
    def spacial_compression_encode(self):
        return 8


class DiffSynthCnetPatch:
    inits = 0

    def __init__(self, model_patch, vae, image, strength, inpaint_image=None, mask=None):
        type(self).inits += 1
        self.model_patch, self.vae, self.image, self.strength = model_patch, vae, image, strength
        self.inpaint_image, self.mask = inpaint_image, mask
        self.encoded_image = torch.arange(image.shape[0] * 4 * (image.shape[1] // 8) * (image.shape[2] // 8),
                                          dtype=torch.float32).reshape(image.shape[0], 4, image.shape[1] // 8, image.shape[2] // 8)
        self.encoded_image_size = (image.shape[1], image.shape[2])


class UnrelatedPatch:
    def __init__(self):
        self.image = torch.zeros(1, 8, 8, 3)


class FakeModel:
    def __init__(self, patches):
        self.model_options = {"transformer_options": {"patches": patches}}

    def clone(self):
        return FakeModel({k: list(v) for k, v in self.model_options["transformer_options"]["patches"].items()})


class Unclonable:
    model_options = {}

    def clone(self):
        raise RuntimeError("no clone")


def _setup():
    img = torch.rand(1, 96, 128, 3)
    p = DiffSynthCnetPatch("mp", FakeVAE(), img, 0.7)
    model = FakeModel({"double_block": [p, UnrelatedPatch()], "single_block": [p]})
    return model, p, img


REGION, CANVAS = (100, 40, 420, 300), (512, 384)


@pytest.mark.parametrize("latent_crop", [False, True])
def test_patch_is_cropped_inside_and_restored_after(latent_crop):
    model, p, img = _setup()
    lat = p.encoded_image.clone()
    with MP.cropped_model_patches(model, REGION, CANVAS, latent_crop=latent_crop) as m:
        assert m is not model
        x1, y1, x2, y2 = MP.scale_region(REGION, CANVAS, (128, 96))
        assert torch.equal(p.image, img[:, y1:y2, x1:x2, :])
        assert p.encoded_image_size == (y2 - y1, x2 - x1)
        if latent_crop:
            assert torch.equal(p.encoded_image, lat[:, :, y1 // 8:y2 // 8, x1 // 8:x2 // 8])
    assert torch.equal(p.image, img) and torch.equal(p.encoded_image, lat) and p.encoded_image_size == (96, 128)


def test_patch_restored_when_the_sampler_raises_and_unclonable_model_passes_through():
    model, p, img = _setup()
    with pytest.raises(KeyError):
        with MP.cropped_model_patches(model, REGION, CANVAS):
            raise KeyError("sampler failed")
    assert torch.equal(p.image, img)
    u = Unclonable()
    with MP.cropped_model_patches(u, REGION, CANVAS) as m:
        assert m is u


def test_patch_shared_by_two_blocks_is_cropped_once():
    model, p, _ = _setup()
    n0 = DiffSynthCnetPatch.inits
    with MP.cropped_model_patches(model, REGION, CANVAS):
        assert DiffSynthCnetPatch.inits == n0 + 1        # re-initialised once although registered twice


def _seen(ctx):
    torch.manual_seed(0)
    model, p, img = _setup()
    with ctx(model):
        seen = (p.image.clone(), p.encoded_image.clone(), tuple(p.encoded_image_size))
    return seen, p, img


def reference_crop_model_cond(latent_crop, region, canvas):
    ref_loader.load()
    R = sys.modules[ref_loader.PKG + ".utils.crop_model_patch"]
    seen, _, _ = _seen(lambda m: R.crop_model_cond(m, region, canvas, canvas, (544, 544), latent_crop=latent_crop))
    return fingerprint(seen)


@pytest.mark.parametrize("latent_crop", [False, True])
@pytest.mark.parametrize("region,canvas", [(REGION, CANVAS), ((0, 0, 544, 544), (1300, 1100)), ((724, 524, 1300, 1100), (1300, 1100))])
def test_matches_reference_crop_model_cond(latent_crop, region, canvas):
    seen, p, img = _seen(lambda m: MP.cropped_model_patches(m, region, canvas, latent_crop=latent_crop))
    assert torch.equal(p.image, img)
    want = reference_fingerprints("test_model_patch")["crop_model_cond"][repr((latent_crop, region, canvas))]
    got = fingerprint(seen)
    assert got["tuple"][0] == want["tuple"][0]
    assert got["tuple"][1] == want["tuple"][1]
    assert got["tuple"][2] == want["tuple"][2]
