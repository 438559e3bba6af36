"""Generate tests/golden/* by RUNNING THE REAL REFERENCE from /root/reference.

Run in the build container only:   python oracle/gen_golden.py
Outputs (committed, small):
  tests/golden/geometry.json      crop windows / process sizes from the reference's
                                  extract_batch_tile_with_padding + calculate_tiles
  tests/golden/single_*.npz       u8 outputs of the reference's process_single_gpu with
                                  the T0 denoiser (inputs are regenerated from seeds)
  tests/golden/prims.npz          create_tile_mask windows and the window blend_tile wrote (inputs from a seed)
  tests/golden/mask_crop.npz      crop_mask outputs (conditioning masks cut to a tile), u8
  tests/golden/static_ref_index.json   the reference's multi-worker static mode run over HTTP here: the tile
                                  assignment each run ended up with + SHA-256 of the master's u8 result

Test infrastructure only (see oracle/usdu_oracle.py header).
"""
from __future__ import annotations

import hashlib
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_loader  # noqa: E402
import usdu_oracle as orc  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


sys.path.insert(0, os.path.join(os.path.dirname(HERE), "tests"))
from inputs import MASK_CROP_CASES, STATIC_REF_CASES, make_input, make_mask, sweep_cases, sweep_sampler  # noqa: E402  (shared with the tests)


def torch_t0(seed_unused=None):
    cache = {}

    def fn(pixels: torch.Tensor, seed: int, denoise: float) -> torch.Tensor:
        d = float(np.float32(denoise))
        omd = float(np.float32(1.0) - np.float32(denoise))
        key = (tuple(pixels.shape), int(seed))
        if key not in cache:
            cache[key] = torch.from_numpy(orc.t0_noise(seed, tuple(pixels.shape)))
        y = pixels * omd + cache[key] * d
        return torch.clamp(y, 0.0, 1.0)

    return fn


GEOMETRY_CASES = [
    # W, H, tile_w, tile_h, padding, uniform
    (512, 512, 256, 256, 32, True),
    (7680, 4320, 512, 512, 32, True),
    (3840, 2160, 512, 512, 32, True),
    (1600, 1200, 512, 512, 32, True),
    (1300, 1100, 512, 512, 32, True),
    (1300, 1100, 512, 512, 32, False),
    (1000, 900, 256, 256, 16, True),
    (1000, 900, 256, 384, 64, True),
    (1000, 900, 256, 384, 64, False),
    (777, 333, 128, 64, 8, True),
    (777, 333, 128, 64, 0, False),
    (100, 90, 128, 128, 32, True),
    (100, 90, 128, 128, 32, False),
    (640, 640, 500, 508, 24, True),     # round_to_multiple banker's cases
    (640, 640, 516, 524, 24, False),
    (2048, 2048, 1024, 1024, 256, True),
    (300, 260, 128, 128, 16, True),
    (200, 168, 64, 64, 8, False),
]

SINGLE_CASES = [
    # name, kind, seed, B, H, W, tile_w, tile_h, padding, blur, uniform, denoise, dseed
    ("cfg1", "noise", 0, 1, 512, 512, 256, 256, 32, 8, True, 0.5, 123),
    ("odd_b2", "noise", 1, 2, 260, 300, 128, 128, 16, 16, True, 0.5, 7),
    ("nonuniform", "smooth", 2, 1, 168, 200, 64, 64, 8, 4, False, 0.35, 11),
    ("upsample", "noise", 3, 1, 90, 100, 128, 128, 32, 8, True, 0.5, 5),
    ("checker", "checker", 0, 1, 200, 232, 96, 80, 16, 8, True, 0.25, 9),
    ("blur0", "smooth", 4, 1, 160, 160, 64, 64, 8, 0, True, 0.5, 3),
    ("pad0", "noise", 5, 1, 160, 192, 64, 64, 0, 6, True, 0.5, 3),
    ("b5_video", "smooth", 6, 5, 136, 168, 64, 64, 16, 8, True, 0.35, 42),
]


def gen_mask_crop():
    """tests/golden/mask_crop.npz: the reference's crop_mask (utils/usdu_utils.py:415-442) on seeded masks."""
    ref_loader.load()
    U = sys.modules[ref_loader.PKG + ".utils.usdu_utils"]
    out = {}
    for (name, kind, seed, B, (Hm, Wm), region, canvas, tile) in MASK_CROP_CASES:
        m = torch.from_numpy(make_mask(kind, seed, B, Hm, Wm))
        d = {"mask": m.clone()}
        U.crop_mask(d, region, canvas, canvas, tile, 0, 0)
        res = d["mask"].numpy()
        q = np.round(res * 255).astype(np.uint8)
        assert np.array_equal(q.astype(np.float32) / np.float32(255), res)
        out[name] = q
        print("mask_crop", name, q.shape, hashlib.sha256(q.tobytes()).hexdigest()[:16])
    np.savez_compressed(os.path.join(OUT, "mask_crop.npz"), **out)


def gen_static_ref():
    """tests/golden/static_ref_index.json: the reference's multi-worker static mode, really run (master +
    workers over aiohttp with its PNG transport, oracle/ref_static_run.py): per case the tile assignment
    that happened (the workers pull tile ids, so it is recorded, not chosen) and the SHA-256 of the
    master's u8 result (the images are seeded noise -- incompressible -- so only the digest is stored)."""
    import ref_static_run
    index = []
    for (name, kind, seed, B, H, W, tile, pad, blur, uni, n_workers, dseed, den) in STATIC_REF_CASES:
        img = make_input(kind, seed, B, H, W)
        res, asg = ref_static_run.run_static(img, n_workers, tile, pad, blur, uni, dseed, den, master_delay=0.25)
        out = np.round(res * 255).astype(np.uint8)
        assert np.array_equal(out.astype(np.float32) / np.float32(255), res)
        replay = orc.replay_static(img, orc.make_t0_denoiser(dseed, den), tile, tile, pad, blur, uni, asg)
        assert np.array_equal(replay, res), f"{name}: replay_static differs from the reference"
        index.append({"name": name, "kind": kind, "seed": seed, "B": B, "H": H, "W": W, "tile": tile, "padding": pad,
                      "mask_blur": blur, "uniform": uni, "denoise_seed": dseed, "denoise": den, "assignment": asg,
                      "sha256": hashlib.sha256(out.tobytes()).hexdigest()})
        print("static_ref", name, asg, index[-1]["sha256"][:16])
    with open(os.path.join(OUT, "static_ref_index.json"), "w") as f:
        json.dump({"generator": "oracle/gen_golden.py (oracle/ref_static_run.py)", "reference": "a91f9fb", "cases": index}, f, indent=1)


def gen_sweep_digests():
    """tests/golden/sweep_ref_digests.json: SHA-256 of the REAL reference's process_single_gpu output (u8) for
    every case of the seeded parameter sweep the GPU tests run (tests/inputs.py sweep_cases)."""
    node, fake_nodes = ref_loader.make_reference_node()
    digests = {}
    for (i, kind, B, H, W, tw, th, pad, blur, uni) in sweep_cases():
        seed, den = sweep_sampler(i)
        fake_nodes.fn = torch_t0()
        img = make_input(kind, i, B, H, W)
        (res,) = node.process_single_gpu(torch.from_numpy(img), None, [[torch.zeros(1, 77, 8), {}]],
                                         [[torch.zeros(1, 77, 8), {}]], None, seed, 20, 8.0, "euler", "normal", den,
                                         tw, th, pad, blur, uni, False)
        out = np.round(res.numpy() * 255).astype(np.uint8)
        assert np.array_equal(out.astype(np.float32) / np.float32(255), res.numpy())
        digests[str(i)] = hashlib.sha256(out.tobytes()).hexdigest()
        print("sweep", i, kind, B, H, W, tw, th, pad, blur, uni, digests[str(i)][:16], flush=True)
    with open(os.path.join(OUT, "sweep_ref_digests.json"), "w") as f:
        json.dump({"generator": "oracle/gen_golden.py", "reference": "a91f9fb", "digests": digests}, f, indent=1)


def main():
    os.makedirs(OUT, exist_ok=True)
    if "--sweep-only" in sys.argv:
        return gen_sweep_digests()
    if "--mask-crop-only" in sys.argv:
        return gen_mask_crop()
    if "--static-ref-only" in sys.argv:
        return gen_static_ref()
    gen_mask_crop()
    gen_static_ref()
    gen_sweep_digests()
    node, fake_nodes = ref_loader.make_reference_node()
    fake_nodes.fn = torch_t0()

    # ---- geometry -----------------------------------------------------------------
    geo = []
    for (W, H, tw0, th0, pad, uni) in GEOMETRY_CASES:
        tw, th = node.round_to_multiple(tw0), node.round_to_multiple(th0)
        tiles = node.calculate_tiles(W, H, tw, th, uni)
        img = torch.zeros(1, 1, 1, 3).expand(1, H, W, 3)
        rows = []
        for (x, y) in tiles:
            t, x1, y1, ew, eh = node.extract_batch_tile_with_padding(img, x, y, tw, th, pad, uni)
            rows.append([x, y, x1, y1, ew, eh, int(t.shape[2]), int(t.shape[1])])
        geo.append({"W": W, "H": H, "tile_w": tw0, "tile_h": th0, "padding": pad, "uniform": uni,
                    "tw": tw, "th": th, "rows": rows})
        print("geometry", W, H, tw0, th0, pad, uni, len(rows))
    with open(os.path.join(OUT, "geometry.json"), "w") as f:
        json.dump({"generator": "oracle/gen_golden.py", "reference": "a91f9fb", "cases": geo}, f,
                  separators=(",", ":"))

    # ---- primitives: mask windows + blend_tile ----------------------------------------
    from PIL import Image
    rng = np.random.default_rng(1234)
    prims = {}
    pcases = [(300, 260, 128, 128, 128, 128, 16, 16), (300, 260, 0, 0, 128, 128, 8, 32),
              (300, 260, 256, 256, 128, 128, 32, 8), (200, 168, 64, 128, 64, 64, 0, 8)]
    for i, (W, H, x, y, tw, th, blur, pad) in enumerate(pcases):
        mask = node.create_tile_mask(W, H, x, y, tw, th, blur)
        x1, y1, x2, y2, pw, ph = orc.crop_geometry(W, H, x, y, tw, th, pad, True)
        base = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
        tile = rng.integers(0, 256, (ph, pw, 3), dtype=np.uint8)
        out = np.array(node.blend_tile(Image.fromarray(base), Image.fromarray(tile), x1, y1, (x2 - x1, y2 - y1), mask, pad))
        outside = out.copy()
        outside[y1:y2, x1:x2] = base[y1:y2, x1:x2]
        assert np.array_equal(outside, base), "blend_tile changed pixels outside the crop window"
        # base and tile are regenerated from the seed by the test; only the window blend_tile wrote is stored
        prims[f"case{i}_params"] = np.array([W, H, x, y, tw, th, blur, pad, x1, y1, x2, y2, pw, ph])
        prims[f"case{i}_mask"] = np.array(mask)
        prims[f"case{i}_out_window"] = np.ascontiguousarray(out[y1:y2, x1:x2])
        print("prim", i, (W, H, x, y, blur, pad))
    np.savez_compressed(os.path.join(OUT, "prims.npz"), **prims)

    # ---- full single-GPU path -------------------------------------------------------
    index = []
    for (name, kind, seed, B, H, W, tw, th, pad, blur, uni, den, dseed) in SINGLE_CASES:
        img = make_input(kind, seed, B, H, W)
        (res,) = node.process_single_gpu(torch.from_numpy(img), None, [[torch.zeros(1, 77, 8), {}]],
                                         [[torch.zeros(1, 77, 8), {}]], None, dseed, 20, 8.0, "euler",
                                         "normal", den, tw, th, pad, blur, uni, False)
        out = np.round(res.numpy() * 255).astype(np.uint8)
        assert np.array_equal(out.astype(np.float32) / np.float32(255), res.numpy())
        sha = hashlib.sha256(out.tobytes()).hexdigest()
        np.savez_compressed(os.path.join(OUT, f"single_{name}.npz"), out=out)
        index.append({"name": name, "kind": kind, "seed": seed, "B": B, "H": H, "W": W, "tile_w": tw,
                      "tile_h": th, "padding": pad, "mask_blur": blur, "uniform": uni, "denoise": den,
                      "denoise_seed": dseed, "sha256": sha})
        print("single", name, sha[:16])
    with open(os.path.join(OUT, "single_index.json"), "w") as f:
        json.dump({"generator": "oracle/gen_golden.py", "reference": "a91f9fb", "cases": index}, f, indent=1)


if __name__ == "__main__":
    main()
