"""Synthetic canvases shared by the golden generator and the tests (values k/255 fp32)."""
import hashlib

import numpy as np
import torch


def fingerprint(obj):
    """JSON-comparable form of a nested result: every tensor / array becomes "shape/dtype/sha256", containers are
    walked (a tuple stays distinct from a list), scalars and strings stay.  What the reference computed is stored in
    this form under tests/golden/reference_fingerprints.json (oracle/gen_reference_fingerprints.py)."""
    if isinstance(obj, torch.Tensor):
        obj = obj.detach().cpu().contiguous().numpy()
    if isinstance(obj, np.ndarray):
        a = np.ascontiguousarray(obj)
        return f"{list(a.shape)}/{a.dtype}/{hashlib.sha256(a.tobytes()).hexdigest()[:32]}"
    if isinstance(obj, dict):
        return {str(k): fingerprint(v) for k, v in sorted(obj.items(), key=lambda kv: str(kv[0]))}
    if isinstance(obj, tuple):
        return {"tuple": [fingerprint(x) for x in obj]}
    if isinstance(obj, list):
        return [fingerprint(x) for x in obj]
    return obj


def reference_fingerprints(test: str) -> dict:
    """What the reference computed for one side-by-side test, keyed by case (tests/golden/reference_fingerprints.json;
    empty while the generator is writing it, so that a test then fails on the missing case)."""
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_fingerprints.json")
    if not os.path.isfile(path):
        return {}
    with open(path) as f:
        return json.load(f)["tests"].get(test, {})


def make_input(kind: str, seed: int, B: int, H: int, W: int) -> np.ndarray:
    if kind == "noise":
        g = torch.Generator().manual_seed(seed)
        x = torch.rand(B, H, W, 3, generator=g)
        return (torch.floor(x * 255) / 255).numpy().astype(np.float32)
    if kind == "smooth":
        g = torch.Generator().manual_seed(seed)
        yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
        base = np.stack([xx / max(W - 1, 1), yy / max(H - 1, 1), (xx + yy) / max(W + H - 2, 1)], -1)
        n = torch.rand(B, H, W, 3, generator=g).numpy() * 0.1
        v = np.clip(base[None] * 0.9 + n, 0, 1)
        return (np.floor(v * 255) / 255).astype(np.float32)
    if kind == "checker":
        yy, xx = np.mgrid[0:H, 0:W]
        c = (((xx // 3) + (yy // 5)) % 2).astype(np.float32)
        img = np.stack([c, 1 - c, c], -1)[None].repeat(B, 0)
        return img.astype(np.float32)
    raise ValueError(kind)


def make_mask(kind: str, seed: int, B: int, H: int, W: int) -> np.ndarray:
    """Conditioning masks fp32 [B, H, W] in [0, 1] (NOT pre-quantised: the truncating cast is part
    of what is tested)."""
    g = torch.Generator().manual_seed(seed)
    if kind == "noise":
        return torch.rand(B, H, W, generator=g).numpy().astype(np.float32)
    if kind == "blob":
        yy, xx = np.mgrid[0:H, 0:W].astype(np.float32)
        out = []
        for b in range(B):
            cx, cy = (0.3 + 0.2 * b) * W, (0.6 - 0.1 * b) * H
            r = np.sqrt((xx - cx) ** 2 + (yy - cy) ** 2) / (0.35 * max(W, H))
            out.append(np.clip(1.2 - r, 0, 1) * (0.9 + 0.1 * torch.rand(H, W, generator=g).numpy()))
        return np.stack(out).astype(np.float32)
    raise ValueError(kind)


# (name, kind, seed, B, (Hm, Wm), region, canvas (W, H), tile (pw, ph)) -- shared by oracle/gen_golden.py and the tests
MASK_CROP_CASES = [
    ("pad_v", "noise", 1, 2, (96, 64), (10, 20, 170, 150), (300, 260), (160, 136)),
    ("interior_1080p", "blob", 2, 1, (135, 240), (480, 440, 1056, 1016), (1920, 1080), (544, 544)),
    ("corner_pad_v", "noise", 3, 1, (64, 64), (0, 0, 300, 200), (512, 512), (304, 208)),
    ("pad_h", "blob", 4, 2, (200, 100), (100, 37, 413, 260), (700, 500), (320, 224)),
    ("tall_pad_h", "noise", 5, 1, (50, 50), (20, 10, 180, 300), (200, 320), (256, 256)),
    ("last_tile_downscale", "noise", 6, 1, (300, 260), (724, 524, 1300, 1100), (1300, 1100), (544, 544)),
    ("mask_is_canvas", "blob", 7, 1, (1100, 1300), (0, 0, 544, 544), (1300, 1100), (544, 544)),
    ("upsample_tile", "noise", 8, 1, (90, 160), (992, 512, 1280, 800), (1280, 800), (544, 544)),
]


# (name, kind, seed, B, H, W, tile, padding, blur, uniform, n_workers, denoise seed, denoise) -- multi-worker jobs run
# through the REAL reference's HTTP static mode by oracle/gen_golden.py (oracle/ref_static_run.py)
STATIC_REF_CASES = [
    ("w1_700x520_t256", "noise", 3, 1, 520, 700, 256, 32, 8, True, 1, 9, 0.5),
    ("w2_1300x1100_t512", "noise", 4, 1, 1100, 1300, 512, 32, 8, True, 2, 11, 0.5),
    ("w1_b5_420x300_t128", "smooth", 5, 5, 300, 420, 128, 16, 8, True, 1, 13, 0.4),
    ("w3_nonuniform_900x640_t256", "noise", 6, 1, 640, 900, 256, 16, 16, False, 3, 15, 0.6),
]


def sweep_cases():
    """Seeded sweep over the node's parameter space on small canvases (tests/test_gpu_sweep.py; the real
    reference's digests for the same cases: tests/golden/sweep_ref_digests.json by oracle/gen_golden.py).
    -> (id, kind, B, H, W, tile_w, tile_h, padding, mask_blur, uniform); input seed = id, T0 seed = 1000 + id,
    denoise = 0.25 + 0.05 * (id % 10)."""
    rng = np.random.default_rng(20260921)
    out = []
    for i in range(40):
        W = int(rng.integers(24, 700))
        H = int(rng.integers(24, 500))
        tw = int(rng.choice([64, 72, 96, 128, 200, 256, 512]))
        th = int(rng.choice([64, 80, 128, 256, 384]))
        pad = int(rng.choice([0, 8, 16, 32, 64, 128]))
        blur = int(rng.choice([0, 1, 4, 8, 16, 40, 97]))
        uniform = bool(rng.integers(0, 2))
        B = int(rng.choice([1, 1, 1, 2, 5]))
        kind = ["noise", "smooth", "checker"][int(rng.integers(0, 3))]
        out.append((i, kind, B, H, W, tw, th, pad, blur, uniform))
    out += [(100, "noise", 1, 64, 48, 512, 512, 32, 8, True),      # canvas << tile: 544 -> 48 needs 68 taps (generic kernels)
            (101, "noise", 1, 37, 1021, 64, 64, 8, 8, True),       # odd width, wide and flat
            (102, "checker", 1, 515, 33, 128, 128, 16, 255, True),  # narrow, blur far larger than the canvas
            (103, "smooth", 17, 96, 120, 64, 64, 16, 8, True)]      # WAN-style 4n+1 frame batch
    return out


def sweep_sampler(i: int):
    return 1000 + i, 0.25 + 0.05 * (i % 10)
