#!/usr/bin/env python
"""bench.py -- megapixels/sec of the USDU tile path (BASELINE.json: "megapixels/sec 4K->8K
SDXL tile-upscale at 1/2/4/8 B200; blend HBM GB/s").

  python bench.py --gpus N --steps K --warmup W              our arm (CUDA kernels)
  python bench.py --impl reference --gpus N --steps K ...    the reference's CPU path (port)
  python bench.py ... --dump-outputs DIR                      also write what the last timed step computed

A step is one full pass of the hot path over one synthetic canvas: quantise -> per wave
(crop+LANCZOS kernel, sampler call, LANCZOS-back+composite kernel) -> dequantise.
Workload (config.workload): configs[1] of BASELINE.json -- 7680x4320x1 canvas, 512-px
tiles, padding 32, mask_blur 8, uniform tiles, 135 tiles.  The sampler is the deterministic
T0 stand-in on BOTH arms (no SDXL weights / ComfyUI offline; BASELINE.md section 3), so the
number isolates tile ops + transport, which is the path this repo replaces.

`value`   : canvas megapixels / device time with the canvas already resident in HBM.
`e2e`     : same metric through the node API (UltimateSDUpscaleDistributed.run) with a
            pinned HOST tensor in and a HOST tensor out -- H2D/D2H inside the timed region.
`roofline`: dominant kernel (seam blend), algorithmic bytes / CUDA-event time per launch.

--dump-outputs DIR writes rank 0's result of the last timed step as DIR/result.npy (fp32 [B,H,W,3]) when it
is at most DUMP_MAX_BYTES, else as a fixed sample: DIR/result_sample.npy (fp32) holds the values at the flat
indices in DIR/result_sample_index.npy (float64), drawn from a generator seeded with 0.  The inputs are seeded,
so two builds run with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (B, H, W, tile, padding, blur)
    "cfg2_4k_to_8k_sdxl_512px": (1, 4320, 7680, 512, 32, 8),
    "cfg1_512_256px": (1, 512, 512, 256, 32, 8),
    "cfg4_16k_256px": (1, 8640, 15360, 256, 32, 8),
    "cfg5_video_17f_4k": (17, 2160, 3840, 512, 32, 8),
}
SEED, DENOISE = 123, 0.5
DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLES = 4 << 20          # sampled values (fp32) + their indices (float64): 48 MiB


def dump_result(out, path: str) -> None:
    """Write one result tensor under `path` (see --dump-outputs in the module docstring)."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    flat = out.detach().reshape(-1)
    if flat.numel() * 4 <= DUMP_MAX_BYTES:
        np.save(os.path.join(path, "result.npy"), out.detach().to(torch.float32).cpu().numpy())
        return
    idx = torch.randint(flat.numel(), (DUMP_SAMPLES,), generator=torch.Generator().manual_seed(0)).sort().values
    vals = flat[idx.to(flat.device)].to(torch.float32).cpu().numpy()
    np.save(os.path.join(path, "result_sample.npy"), vals)
    np.save(os.path.join(path, "result_sample_index.npy"), idx.numpy().astype(np.float64))


def make_canvas_cpu(B, H, W):
    import torch
    g = torch.Generator().manual_seed(0)
    x = torch.rand(B, H, W, 3, generator=g)
    return torch.floor(x * 255) / 255           # values k/255, like an image that went through ComfyUI


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


class NvlinkCounters:
    """NVLink payload bytes of this rank's GPU (NVML field values NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX / _RX summed over the
    links, KiB): read before and after a timed loop -> bytes per step that crossed the link, measured, not modelled."""

    def __init__(self, index: int):
        self.h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = torch.cuda.get_device_properties(index).uuid
            self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            self.nv = pynvml
            self.ids = [(pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF), (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)]
            self.read()
        except Exception:
            self.h = None

    def read(self):
        if self.h is None:
            return None
        try:
            v = self.nv.nvmlDeviceGetFieldValues(self.h, self.ids)
            out = []
            for x in v:
                if x.nvmlReturn != 0:
                    return None
                out.append(int(x.value.ullVal) * 1024)
            return out                       # [tx bytes, rx bytes]
        except Exception:
            return None


def kernel_source_hash() -> str:
    """SHA-256 over the CUDA sources and the C header the library is built from (a stamp that is the same on the build
    container and on the GPU box; the .so itself is rebuilt per box)."""
    import glob
    import hashlib
    h = hashlib.sha256()
    for f in sorted(glob.glob(os.path.join(ROOT, "comfyui-distributed_b200", "csrc", "*.cu*")) + [os.path.join(ROOT, "include", "usdu_b200.h")]):
        h.update(os.path.basename(f).encode())
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def expected_digest(workload: str, world: int):
    """SHA-256 of the u8 result the reference produces for this workload (tests/golden/bench_digests.json, written by
    oracle/gen_bench_digests.py: the REAL reference's process_single_gpu for N = 1 where it was run, the oracle
    otherwise; oracle.replay_static of the recorded assignment for N > 1).  -> (entry, key) or (None, key)."""
    p = os.path.join(ROOT, "tests", "golden", "bench_digests.json")
    key = f"{workload}/n{world}"
    if not os.path.isfile(p):
        return None, key
    db = json.load(open(p))["digests"]
    for src in ("reference", "oracle"):
        if f"{key}/{src}" in db:
            return db[f"{key}/{src}"], f"{key}/{src}"
    return None, key


def result_digest(out) -> str:
    """SHA-256 of a result tensor [B,H,W,3] fp32 (values k/255, any device) as u8."""
    import hashlib
    import torch
    q = torch.round(out.detach().to(torch.float32) * 255).to(torch.uint8).cpu().contiguous()
    return hashlib.sha256(q.numpy().tobytes()).hexdigest()


# --------------------------------------------------------------------------------------
# CPU baseline: the reference's OWN code (oracle/make_ref.py bundles its sources into the git-ignored oracle/_ref/
# at build time; oracle/ref_loader.py loads them under ComfyUI stand-ins), on a bounded sample of the workload
# --------------------------------------------------------------------------------------
def _oracle_path():
    p = os.path.join(ROOT, "oracle")
    if p not in sys.path:
        sys.path.insert(0, p)


def _t0_torch():
    """The T0 sampler stand-in on torch CPU tensors (same arithmetic as denoise.T0Denoiser / oracle.make_t0_denoiser)."""
    import numpy as np
    import torch
    cache = {}

    def fn(pixels, seed, denoise):
        key = (tuple(pixels.shape), int(seed))
        if key not in cache:
            cache[key] = torch.rand(tuple(pixels.shape), generator=torch.Generator().manual_seed(int(seed)), dtype=torch.float32)
        d = np.float32(denoise)
        return torch.clamp(pixels * float(np.float32(1.0) - d) + cache[key] * float(d), 0.0, 1.0)

    return fn


def reference_available() -> bool:
    _oracle_path()
    import make_ref
    return bool(make_ref.staged_root())


_REF_FIXED = {}


def real_reference_sample(workload: str, n_tiles: int):
    """N = 1: the reference's process_single_gpu (upscale/modes/single_gpu.py:8-72), unmodified, on the FIRST n_tiles tiles
    of the full canvas (its calculate_tiles is wrapped on the node object; every per-tile cost -- full-canvas mask, full-canvas
    tensor<->PIL conversions, full-canvas RGBA composite -- is the real one).  Job time = fixed part (a 0-tile run: the
    conversions around the loop) + per-tile time x all tiles."""
    import torch
    _oracle_path()
    import ref_loader
    B, H, W, tile, pad, blur = WORKLOADS[workload]
    img = make_canvas_cpu(B, H, W)
    node, fake_nodes = ref_loader.make_reference_node()
    fake_nodes.fn = _t0_torch()
    full = node.calculate_tiles
    total = len(full(W, H, node.round_to_multiple(tile), node.round_to_multiple(tile), True))
    cond = [[torch.zeros(1, 77, 8), {}]]

    def run(k):
        node.calculate_tiles = lambda *a, **kw: full(*a, **kw)[:k]
        t0 = time.perf_counter()
        node.process_single_gpu(img, None, cond, cond, None, SEED, 20, 8.0, "euler", "normal", DENOISE, tile, tile, pad, blur, True, False)
        return time.perf_counter() - t0

    if workload not in _REF_FIXED:
        _REF_FIXED[workload] = run(0)                  # measured once per process
    fixed = _REF_FIXED[workload]
    n_tiles = max(1, min(n_tiles, total))
    wall = run(n_tiles)
    per_tile = max(wall - fixed, 1e-9) / n_tiles
    est = fixed + per_tile * total
    mp = B * H * W / 1e6
    return {"value": mp / est, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "reference",
            "sample": f"the reference's own process_single_gpu on the first {n_tiles} of {total} tiles of {workload} (full canvas, T0 sampler): "
                      f"fixed {fixed:.1f}s + {per_tile:.2f}s/tile -> {est:.0f}s/job extrapolated; Pillow is single-threaded, torch ops use `cores` threads",
            "host_cpus": os.cpu_count(), "source": f"oracle/_ref (oracle/make_ref.py) via oracle/ref_loader.py: {ref_loader.REF_ROOT}"}


def real_reference_static_sample(workload: str, participants: int, tiles_per_participant: int):
    """N > 1: the reference's static mode really run -- master + N-1 workers, its own HTTP routes on an aiohttp server on
    127.0.0.1, its PNG-multipart transport, its pull queue and its sorted final blend (upscale/modes/static.py:191-570,
    upscale/worker_comms.py:16-188) -- on a job of the first N x tiles_per_participant tiles of the full canvas.  Every phase
    of that mode is linear in the number of tiles, so job time = fixed + (sample - fixed) x all tiles / sample tiles."""
    import torch
    _oracle_path()
    import ref_static_run
    import usdu_oracle as orc
    B, H, W, tile, pad, blur = WORKLOADS[workload]
    img = make_canvas_cpu(B, H, W).numpy()
    total = len(orc.make_plan(W, H, tile, tile, pad, True)[2])
    k = max(1, min(participants * tiles_per_participant, total))
    t0 = time.perf_counter()
    _, asg = ref_static_run.run_static(img, participants - 1, tile, pad, blur, True, SEED, DENOISE, job_id=f"bench{time.time_ns()}",
                                       timeout=1500.0, max_tiles=k)
    wall = time.perf_counter() - t0
    fixed = min(0.25 * wall, 2.0 * B * H * W * 3 * 4 / 1e9)          # tensor<->PIL conversions around the loop (~2 s per GB)
    est = fixed + (wall - fixed) * total / k
    mp = B * H * W / 1e6
    return {"value": mp / est, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "reference", "participants": participants,
            "sample": f"the reference's own static mode (master + {participants - 1} workers as threads of one process -- Pillow and torch "
                      f"release the GIL in their C loops --, real aiohttp routes + PNG transport on 127.0.0.1) on the first {k} of {total} "
                      f"tiles of {workload}: {wall:.1f}s, tiles per participant {[len(a) for a in asg]} -> {est:.0f}s/job extrapolated linearly",
            "host_cpus": os.cpu_count(), "source": f"oracle/_ref via oracle/ref_static_run.py: {ref_static_run.REF_ROOT}"}


def cpu_port_sample(workload: str, budget_s: float):
    """Fallback when the reference bundle is absent: oracle/ref_port.py, the port with the reference's cost structure."""
    import torch
    _oracle_path()
    import ref_port
    B, H, W, tile, pad, blur = WORKLOADS[workload]
    img = make_canvas_cpu(B, H, W)
    t = {}
    t0 = time.perf_counter()
    ref_port.process_single(img, ref_port.torch_t0(SEED, DENOISE), tile, tile, pad, blur, True,
                            time_budget_s=budget_s, timer_out=t)
    wall = time.perf_counter() - t0
    done, total = t["tiles_done"], t["tiles_total"]
    fixed = t.get("q0", 0.0) + t.get("result", 0.0)
    per_tile = (wall - fixed) / done
    est = fixed + per_tile * total                       # extrapolated full-job time
    mp = B * H * W / 1e6
    return {"value": mp / est, "unit": "MP/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"first {done} of {total} tiles of {workload} on the full canvas (oracle/ref_port.py: reference's "
                      f"full-canvas Pillow ops, T0 sampler); fixed {fixed:.1f}s + {per_tile:.2f}s/tile -> {est:.0f}s/job extrapolated",
            "host_cpus": os.cpu_count(), "phases_s": {k: round(v, 3) for k, v in t.items() if isinstance(v, float)}}


def cpu_baseline_sample(workload: str, n_tiles: int, budget_s: float):
    return real_reference_sample(workload, n_tiles) if reference_available() else cpu_port_sample(workload, budget_s)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores, one bounded sample
    (whatever --steps says: a sample is tens of seconds to minutes of CPU work).  N == 1: process_single_gpu.
    N > 1: the N-participant HTTP + PNG static mode.  Falls back to the cost-faithful port (oracle/ref_port*.py) only
    when oracle/_ref is missing."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = args.workload
    B, H, W, tile, pad, blur = WORKLOADS[workload]
    mp = B * H * W / 1e6
    steps = max(1, args.steps)
    # every step is a bounded sample; the whole run stays within a few minutes whatever K is: the tiles of the sample are
    # divided over the steps, and the loop stops taking new samples after 150 s (steps actually taken are reported)
    vals, detail, t_start = [], None, time.perf_counter()
    for i in range(steps):
        if vals and time.perf_counter() - t_start > 150.0:
            break
        if reference_available():
            if args.gpus == 1:
                detail = real_reference_sample(workload, max(1, args.ref_tiles // steps))
            else:
                detail = real_reference_static_sample(workload, args.gpus, args.ref_tiles_per_participant)
        elif args.gpus == 1:
            detail = cpu_port_sample(workload, max(3.0, min(args.ref_budget, 150.0 / steps)))
        else:
            _oracle_path()
            import ref_port_http
            detail = ref_port_http.bench_sample(WORKLOADS[workload], SEED, DENOISE, participants=args.gpus,
                                                tiles_per_participant=args.ref_tiles_per_participant)
        vals.append(detail["value"])
    detail = dict(detail, value=sum(vals) / len(vals), samples=len(vals))
    v = detail["value"]
    line = {"impl": "reference", "metric": "megapixels/sec", "value": v, "unit": "MP/s", "n_gpus": args.gpus,
            "steps": len(vals), "requested_steps": steps, "warmup": 0, "ms_per_step": mp / v * 1e3, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload, "canvas": [B, H, W], "tile": tile, "padding": pad, "mask_blur": blur,
                       "denoiser": "T0 deterministic stand-in", "timing": "wall clock, extrapolated from a bounded sample"},
            "cpu_baseline": detail,
            "e2e": {"value": v, "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_4k_to_8k_sdxl_512px", choices=list(WORKLOADS))
    ap.add_argument("--denoiser", default="t0", choices=["t0", "t1"])
    ap.add_argument("--cpu-budget", type=float, default=15.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--ref-budget", type=float, default=20.0)
    ap.add_argument("--ref-tiles-per-participant", type=int, default=3)
    ap.add_argument("--ref-tiles", type=int, default=6, help="tiles of the bounded sample of --impl reference at N = 1")
    ap.add_argument("--cpu-tiles", type=int, default=3, help="tiles of the bounded cpu_baseline sample of our arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-t1", action="store_true", help="skip the supplementary SDXL-cost (T1) measurement")
    ap.add_argument("--semantics", default="static", choices=["static", "exact"],
                    help="N > 1: the reference's static mode (default, the headline) or the cooperative single-GPU DAG "
                         "(dist.upscale_exact: bit-identical to N = 1 at any world size; device-resident line only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step under DIR as .npy (a seeded sample when it is large)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs needs the CUDA arm: --impl reference times a bounded sample of the job")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as td
    from __graft_entry__ import load_package
    load_package()
    from comfyui_distributed_b200 import dist as udist
    from comfyui_distributed_b200 import engine
    from comfyui_distributed_b200 import planner as planner_mod
    from comfyui_distributed_b200.denoise import T0Denoiser
    from comfyui_distributed_b200.nodes import UltimateSDUpscaleDistributed
    from comfyui_distributed_b200.testing import SyntheticSDXLModel, T0Model

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the USDU kernels have no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        td.init_process_group("nccl", device_id=dev)
    if args.gpus != world:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run --nproc-per-node {args.gpus}")

    B, H, W, tile, pad, blur = WORKLOADS[args.workload]
    mp = B * H * W / 1e6
    host = make_canvas_cpu(B, H, W).pin_memory()
    img = host.to(dev)
    if args.denoiser == "t0":
        model = T0Model()
        den = T0Denoiser(SEED, DENOISE)
        den_name = "T0 deterministic stand-in (x*(1-d)+rand(seed)*d), one fused elementwise kernel on device"
    else:
        model = SyntheticSDXLModel(device=dev)
        den = model.as_usdu_denoiser(steps=20, denoise=DENOISE)
        den_name = "T1 synthetic SDXL-cost torch module (bf16, 20 steps x2 cfg)"
    node = UltimateSDUpscaleDistributed()

    def barrier():
        if world > 1:
            td.barrier()
        torch.cuda.synchronize()

    exact = world > 1 and args.semantics == "exact"

    def step_device(stats=None):
        if exact:
            return udist.upscale_exact(img, den, tile, tile, pad, blur, True, stats=stats)
        if world > 1:
            return udist.upscale_static(img, den, tile, tile, pad, blur, True, stats=stats)
        return engine.upscale_single(img, den, tile, tile, pad, blur, True, stats=stats)

    def step_e2e():
        if exact:                    # the node API has no switch for it: the supplementary line reports the device-resident job only
            return step_device()
        return node.run(host, model, None, None, None, SEED, 20, 8.0, "euler", "normal", DENOISE, tile, tile, pad, blur,
                        True, False, multi_job_id="bench" if world > 1 else "")[0]

    # ---- device-resident metric -------------------------------------------------------
    # ---- device-resident metric: K steps between two events, nothing else in the stream -------------
    def timed(fn, steps):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=dev)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item()) / steps

    # ---- parity first: one untimed step per arm; rank 0's result against the committed digest of the reference --------
    parity = {"checked": False, "match": None, "why": "no digest for this workload / sampler"}
    exp, exp_key = expected_digest(args.workload, 1 if exact else world)
    if args.denoiser == "t0" and exp is not None:
        out_dev, out_e2e = step_device(), step_e2e()
        barrier()
        ok = 1
        if rank == 0:
            got = {"device_arm": result_digest(out_dev), "e2e_arm": result_digest(out_e2e)}
            plan0 = planner_mod.get_plan(W, H, tile, tile, pad, blur, True)
            same_asg = world == 1 or exact or [list(map(int, a)) for a in plan0.partition(world)] == exp.get("assignment")
            match = same_asg and all(v == exp["sha256"] for v in got.values())
            parity = {"checked": True, "match": bool(match), "source": f"tests/golden/bench_digests.json:{exp_key} ({exp['how']})",
                      "expected": exp["sha256"], **got}
            if not same_asg:
                parity["why"] = "planner.partition differs from the assignment the digest was generated for"
            ok = int(match)
        del out_dev, out_e2e
        if world > 1:
            # the other two multi-rank paths of SURVEY.md 8f, checked here so that every N-GPU bench run proves them:
            # (f2) exact mode == the 1-GPU digest at this world size; (f1) the collector's order and quantisation asymmetry
            exp1, _ = expected_digest("cfg1_512_256px", 1)
            B1, H1, W1, t1, p1, b1 = WORKLOADS["cfg1_512_256px"]
            img1 = make_canvas_cpu(B1, H1, W1).to(dev)
            ex = udist.upscale_exact(img1, den, t1, t1, p1, b1, True)
            from comfyui_distributed_b200.nodes import DistributedCollectorNode
            g = torch.Generator().manual_seed(100 + rank)
            mine = torch.rand(1 + rank % 2, 64, 48, 3, generator=g)
            ids = [f"rank{r}" for r in range(1, world)]
            got_c, _ = DistributedCollectorNode().run(mine, multi_job_id="bench", is_worker=rank != 0, enabled_worker_ids=json.dumps(ids),
                                                      worker_id="" if rank == 0 else f"rank{rank}")
            if rank == 0:
                parts = [mine]
                for r in range(1, world):
                    w = torch.rand(1 + r % 2, 64, 48, 3, generator=torch.Generator().manual_seed(100 + r))
                    parts.append((w * 255).to(torch.uint8).to(torch.float32) / 255)         # worker images travel as trunc(255 x)
                parity["exact_mode_cfg1_equals_1gpu_digest"] = bool(exp1 is not None and result_digest(ex) == exp1["sha256"])
                parity["collector_order_and_values"] = bool(torch.equal(got_c, torch.cat(parts, 0)))
                ok = int(ok and parity["exact_mode_cfg1_equals_1gpu_digest"] and parity["collector_order_and_values"])
                parity["match"] = bool(ok)
            del ex
        flag = torch.tensor([ok], device=dev)
        if world > 1:
            td.broadcast(flag, 0)
        if int(flag.item()) == 0:
            if rank == 0:
                print(json.dumps({"error": "parity mismatch: the result differs from the reference's digest; nothing timed",
                                  "parity": parity}))
            if world > 1:
                td.destroy_process_group()
            sys.exit(3)

    for _ in range(max(args.warmup, 3)):
        step_device()
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    stats = {}
    nvl = NvlinkCounters(local) if world > 1 else None
    nvl0 = nvl.read() if nvl else None
    last = []

    def timed_step():
        out = step_device(stats)
        if args.dump_outputs:
            last[:] = [out]

    ms_step = timed(timed_step, args.steps)
    nvl1 = nvl.read() if nvl else None
    nvlink = None
    if nvl0 is not None and nvl1 is not None:
        t = torch.tensor([(nvl1[0] - nvl0[0]) / args.steps, (nvl1[1] - nvl0[1]) / args.steps], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(t) for _ in range(world)]
        td.all_gather(allr, t)
        nvlink = {"source": "NVML NVLINK_THROUGHPUT_DATA_TX/RX over the timed device loop, per step",
                  "tx_MB_per_step_by_rank": [round(float(a[0]) / 1e6, 2) for a in allr],
                  "rx_MB_per_step_by_rank": [round(float(a[1]) / 1e6, 2) for a in allr]}
        rx0 = float(allr[0][1])
        if rx0 > 0:
            nvlink["master_rx_GBps_if_spread_over_the_step"] = round(rx0 / (ms_step * 1e-3) / 1e9, 1)
    # (the sampler keeps running through the per-kernel and end-to-end timed loops below: K steps of a
    # 1.3 ms job are over before nvidia-smi's first 100 ms tick)
    stats["gpu_launches"] = stats.get("gpu_launches", 0) // args.steps        # per step
    stats["algo_bytes"] = stats.get("algo_bytes", 0) // args.steps

    # ---- per-kernel time of the dominant kernels, in situ -------------------------------------------
    # N == 1: the wave loop is a CUDA graph; event-record nodes between its ~95 kernels cost ~0.5 ms per
    # step (measured: 1.46 vs 2.01 ms), so the kernels are timed by DIFFERENCING instead: the same K
    # steps with a graph that lacks the blend (resp. crop) launches; the difference is what the kernel
    # costs where it runs (launch latency and cache state included).  N > 1: CUDA events around every
    # launch (the final ordered blend is an eager launch there).
    kern = {}
    if world == 1 and getattr(den, "cuda_graph_safe", False) and engine.USE_CUDA_GRAPHS:
        plan = planner_mod.get_plan(W, H, tile, tile, pad, blur, True)
        n_waves = len(plan.waves())
        wl_bytes = {"crop_resize": 0, "blend": 0}
        for w in plan.waves():
            cw, offs_w, _ = plan.crop_worklist(w, B)
            wl_bytes["crop_resize"] += cw.algo_bytes * B
            wl_bytes["blend"] += plan.blend_worklist(w, offs_w, 4, None, B).algo_bytes * B
        # Kernel DURATIONS are taken in the plain level loop (schedule "waves": one kernel at a time).  The timed step above
        # runs the default schedule (split_crop), where the early crop jobs of level k+1 overlap blend(k): differencing THAT
        # graph would credit the blend with the crop time it hides (measured: 12.7 instead of 14.8 us per launch).
        timed_schedule = engine.SCHEDULE
        engine.SCHEDULE = "waves"
        try:
            fn_full = lambda: engine.upscale_single(img, den, tile, tile, pad, blur, True)
            for _ in range(3):
                fn_full()
            ms_waves = timed(fn_full, args.steps)
            for name in ("blend", "crop_resize"):
                skip = ("blend",) if name == "blend" else ("crop",)
                fn = lambda: engine.upscale_single(img, den, tile, tile, pad, blur, True, _skip=skip)
                for _ in range(3):
                    fn()
                ms_without = timed(fn, args.steps)
                d_ms = max(ms_waves - ms_without, 1e-6)
                kern[name] = {"launches": n_waves, "ms": d_ms, "bytes": wl_bytes[name], "gbps": wl_bytes[name] / (d_ms * 1e-3) / 1e9,
                              "avg_us": d_ms * 1e3 / n_waves}
        finally:
            engine.SCHEDULE = timed_schedule
        timing_note = (f"differencing in the plain level loop (schedule waves, {ms_waves:.4f} ms per step; the timed step runs "
                       f"schedule {timed_schedule}, where the early crop jobs of the next level overlap the blend): {args.steps} "
                       f"steps of the full wave graph vs the same graph without this kernel's {n_waves} launches, CUDA events "
                       "around each batch (no event nodes inside the graph)")
    else:
        prof = engine.KernelProfile()
        engine.PROFILE = prof
        for _ in range(2):
            prof.begin_step()
            step_device()
        barrier()
        engine.PROFILE = None
        kern = prof.summary()
        timing_note = "CUDA events around every launch of one step after the timed region"

    # ---- the two tile kernels in isolation on a machine-filling work list: ALL tiles in one launch (the shape of the
    # static-mode final composite), CUDA events around each launch; the in-situ numbers above are 31 small launches
    isolated = None
    if world == 1:
        plan_i = planner_mod.get_plan(W, H, tile, tile, pad, blur, True)
        dp_i = engine.DevicePlan.get(plan_i, dev)
        cv = engine.Canvas(dp_i, B).load(img)
        ids_i = list(range(len(plan_i.tiles)))
        buf_i, offs_i = cv.crop(ids_i)
        src_i = torch.rand(buf_i.numel(), device=dev)

        def med_us(fn, reps=7):
            for _ in range(2):
                fn()
            ts = []
            for _ in range(reps):
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record(); fn(); b_.record(); torch.cuda.synchronize()
                ts.append(a_.elapsed_time(b_) * 1e3)
            return sorted(ts)[len(ts) // 2]

        cb = dp_i.crop_list(tuple(ids_i), B, cv.path_crop)[0].algo_bytes * B
        bb = dp_i.blend_list(tuple(ids_i), offs_i, False, cv.path_blend, B)[0].algo_bytes * B
        t_c = med_us(lambda: cv.crop(ids_i, out=buf_i))
        t_b = med_us(lambda: cv.blend(ids_i, src_i, offs_i))
        isolated = {"what": f"all {len(ids_i)} tiles in ONE launch, eager, CUDA events, median of 7 (inputs larger than L2)",
                    "blend": {"us": round(t_b, 1), "GBps": round(bb / t_b / 1e3, 1), "frac": round(bb / t_b / 1e3 / measured_peak_gbs()[0], 4), "algorithmic_MB": round(bb / 1e6, 1)},
                    "crop_resize": {"us": round(t_c, 1), "GBps": round(cb / t_c / 1e3, 1), "frac": round(cb / t_c / 1e3 / measured_peak_gbs()[0], 4), "algorithmic_MB": round(cb / 1e6, 1)}}
        del cv, buf_i, src_i

    # ---- N > 1: where the step goes, per phase, max over ranks (CUDA events at the phase boundaries) -----------------
    phases = None
    if world > 1:
        acc = {}
        for _ in range(5):
            st = {"time_phases": True}
            step_device(st)
            for k_, v_ in st.get("phase_ms", {}).items():
                acc.setdefault(k_, []).append(v_)
        if acc:
            names = list(acc)
            t = torch.tensor([sorted(acc[n_])[len(acc[n_]) // 2] for n_ in names], device=dev)     # median of 5 per rank
            td.all_reduce(t, op=td.ReduceOp.MAX)
            phases = {n_: round(float(v_), 4) for n_, v_ in zip(names, t.tolist())}

    # ---- end to end through the node API (host tensor in, host tensor out) -------------
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(max(args.warmup, 3)):
        out_host = step_e2e()      # keep the result like the timed loop does: the second pinned result
                                   # buffer (a one-time ~150 ms page-locking cost) is created here, not in the timed region
    barrier()
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        out_host = step_e2e()
    e1.record()
    barrier()
    e2e_wall = (time.perf_counter() - t0) * 1e3 / args.steps
    t = torch.tensor([max(e0.elapsed_time(e1) / args.steps, e2e_wall)], device=dev)
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    e2e_ms = float(t.item())
    clk = clocks.stop()
    img_bytes = B * H * W * 3 * 4
    e2e_phases = None
    if world > 1 and not exact:                          # where the end-to-end call goes, per phase, max over ranks
        acc = {}
        for _ in range(5):
            node.time_phases = True
            step_e2e()
            for k_, v_ in ((getattr(node, "last_stats", None) or {}).get("phase_ms") or {}).items():
                acc.setdefault(k_, []).append(v_)
        node.time_phases = False
        if acc:
            names = list(acc)
            t = torch.tensor([sorted(acc[n_])[len(acc[n_]) // 2] for n_ in names], device=dev)
            td.all_reduce(t, op=td.ReduceOp.MAX)
            e2e_phases = {n_: round(float(v_), 4) for n_, v_ in zip(names, t.tolist())}

    # ---- supplementary: the same job with an SDXL-cost sampler (T1), one timed step -----------
    t1_info = None
    if args.denoiser == "t0" and not args.no_t1:
        t1_model = SyntheticSDXLModel(device=dev)
        t1_den = t1_model.as_usdu_denoiser(steps=20, denoise=DENOISE)

        def step_t1():
            if world > 1:
                return udist.upscale_static(img, t1_den, tile, tile, pad, blur, True)
            return engine.upscale_single(img, t1_den, tile, tile, pad, blur, True)

        torch.cuda.empty_cache()
        step_t1()                                       # warm-up (cuDNN / SDPA autotune)
        barrier()
        e0.record()
        step_t1()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            td.all_reduce(t, op=td.ReduceOp.MAX)
        t1_ms = float(t.item())
        t1_info = {"value": mp / (t1_ms * 1e-3), "unit": "MP/s", "ms_per_step": t1_ms, "steps": 1, "warmup": 1,
                   "denoiser": "T1 synthetic SDXL-cost torch module (random weights, bf16, 20 steps x 2 cfg passes, ~33 TFLOP/tile)",
                   "note": "supplementary: shows the regime the multi-GPU path is built for (sampler-bound); not the headline"}

    if rank != 0:
        if world > 1:
            td.destroy_process_group()
        return
    if args.dump_outputs:
        dump_result(last[0], args.dump_outputs)
    del last

    peak, peak_src = measured_peak_gbs()
    dom = "blend"
    k = kern.get(dom, {"gbps": 0.0, "launches": 0, "avg_us": 0.0, "bytes": 0})
    traffic, traffic_note = None, None
    tp = os.path.join(ROOT, "profiles", "r02_traffic_cfg2.json")
    if os.path.isfile(tp) and world == 1 and args.workload == "cfg2_4k_to_8k_sdxl_512px":
        tj = json.load(open(tp))
        if tj.get("source_hash") == kernel_source_hash():
            traffic = tj["blend"]["dram_bytes_per_launch"]
            traffic_note = (f"ncu dram__bytes_read+write summed over the {tj['blend']['launches']} blend launches of one step "
                            f"({tj['blend']['dram_bytes_per_step'] / 1e6:.1f} MB = {tj['blend']['traffic_over_algorithmic']} x algorithmic), "
                            f"per launch; profiles/r02_traffic_cfg2.json, captured from kernel sources {tj['source_hash']} = the ones running")
        else:
            traffic_note = (f"profiles/r02_traffic_cfg2.json was captured from kernel sources {tj.get('source_hash')}, the library here is built "
                            f"from {kernel_source_hash()}: traffic withheld (re-capture with tools/one_step.py + tools/traffic_summary.py)")
    plan_r = planner_mod.get_plan(W, H, tile, tile, pad, blur, True)
    survey_bytes = sum(6 * t.pw * t.ph + 6 * t.ew * t.eh for t in plan_r.tiles) * B      # SURVEY.md 8(d): u8 canvas r+w, fp16 tiles
    kernel_name = {2: "usdu::mma::blend_mma_kernel (tensor cores: mma.sync.m16n8k32 u8 x 8-bit coefficient limbs)",
                   1: "usdu::fast::blend_fast_kernel", 0: "usdu::blend_kernel (generic)"}[min(plan_r.kernel_path(None), engine.PATH_BLEND)]
    step_us = k["avg_us"] * max(k["launches"], 1)
    roofline = {"bound": "hbm", "kernel": kernel_name, "achieved": round(k["gbps"], 1), "peak": peak,
                "unit": "GB/s", "frac": round(k["gbps"] / peak, 4), "traffic": traffic, "traffic_note": traffic_note,
                "frac_survey_bytes": round(survey_bytes / (step_us * 1e-6) / 1e9 / peak, 4) if (step_us > 0 and world == 1) else None,
                "survey_bytes_per_step": survey_bytes,
                "isolated_full_launch": isolated,
                "peak_source": peak_src,
                "launches_per_step": k["launches"], "avg_launch_us": round(k["avg_us"], 2),
                "algorithmic_bytes_per_step": k["bytes"],
                "timing": timing_note,
                "other_kernels": {n: {"gbps": round(d["gbps"], 1), "avg_us": round(d["avg_us"], 2),
                                      "launches_per_step": d["launches"]} for n, d in kern.items() if n != dom}}
    line = {"metric": "megapixels/sec", "value": mp / (ms_step * 1e-3), "unit": "MP/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": args.workload, "canvas": [B, H, W], "tile": tile, "padding": pad, "mask_blur": blur,
                       "tiles": stats.get("tiles"), "waves": stats.get("waves"), "denoiser": den_name,
                       "semantics": ("exact progressive (single_gpu)" if world == 1 else
                                     "exact progressive on N ranks (dist.upscale_exact: per-wave all-gather, replicated blend)" if exact
                                     else "static replay, fixed partition"),
                       "cuda_graph": bool(engine.USE_CUDA_GRAPHS and getattr(den, "cuda_graph_safe", False)),
                       "schedule": engine.SCHEDULE if world == 1 else None,
                       "transport": stats.get("transport"),
                       "l2": "inputs larger than L2 (canvas 99.5 MB u8 + 398 MB fp32 image per step)"},
            "clocks": clk,
            "e2e": {"value": mp / (e2e_ms * 1e-3), "unit": "MP/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": img_bytes, "d2h_bytes_per_step": img_bytes,
                    "api": "UltimateSDUpscaleDistributed.run(host tensor) -> host tensor",
                    "note": ("upload, kernels and download overlap band by band (engine.HostPipeline)" if world == 1 else
                             "every rank uploads and downloads only its slab (1/N of the rows) over its own PCIe link; the quantised "
                             "slabs are exchanged over NVLink; the result lands in one page-locked shared-memory tensor "
                             "(dist.upscale_static_host); h2d/d2h bytes are the job's totals over all ranks")},
            "gpu_launches": stats.get("gpu_launches", 0) * args.steps,
            "gpu_launches_per_step": stats.get("gpu_launches", 0),
            "parity": parity,
            "roofline": roofline}
    if phases is not None:
        line["phase_ms_max_over_ranks"] = phases
    if nvlink is not None:
        line["nvlink"] = nvlink
    if e2e_phases is not None:
        line["e2e"]["phase_ms_max_over_ranks"] = e2e_phases
    if t1_info is not None:
        line["sdxl_cost_tier"] = t1_info
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_sample(args.workload, args.cpu_tiles, args.cpu_budget)
    print(json.dumps(line))
    if world > 1:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
