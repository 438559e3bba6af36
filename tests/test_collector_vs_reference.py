"""oracle.collector_combine and our audio combination == the reference's own DistributedCollector (worker PNG
round trip, master decode, _reorder_and_combine_tensors, _combine_audio).  What the reference computed is stored
in tests/golden/collector_ref.json and tests/golden/reference_fingerprints.json (oracle/ref_collector.py loads the
reference to regenerate them)."""
import hashlib
import json
import os

import numpy as np
import pytest
import torch

import ref_collector
import usdu_oracle as orc
from inputs import fingerprint, reference_fingerprints

G = os.path.join(os.path.dirname(__file__), "golden")
CASES = json.load(open(os.path.join(G, "collector_ref.json")))["cases"]


def _inputs(case):
    g = torch.Generator().manual_seed(case["seed"])
    H, W = case["H"], case["W"]
    master = torch.rand(case["master_b"], H, W, 3, generator=g)
    workers = {w: torch.rand(b, H, W, 3, generator=g) for w, b in case["workers"]}
    return master, workers


@pytest.mark.parametrize("case", CASES, ids=lambda c: c["name"])
def test_oracle_collector_matches_golden(case):
    master, workers = _inputs(case)
    out = orc.collector_combine(master.numpy(), {w: t.numpy() for w, t in workers.items()}, case["order"], case["delegate"])
    assert hashlib.sha256(np.ascontiguousarray(out, dtype=np.float32).tobytes()).hexdigest() == case["sha256"]
    assert list(out.shape) == case["shape"]


def _audio_cases():
    """200 random piece sets: missing audio, empty waveforms, non-default sample rates, unexpected worker ids."""
    rng = np.random.default_rng(0)

    def piece():
        k = rng.integers(0, 4)
        if k == 0:
            return None
        n = 0 if k == 1 else int(rng.integers(1, 50))
        return {"waveform": torch.from_numpy(rng.random((1, 2, n), dtype=np.float32)), "sample_rate": int(rng.choice([44100, 48000, 22050]))}

    for _ in range(200):
        master = piece()
        ids = ["w1", "w2", "w3", "zz"]
        workers = {w: piece() for w in ids if rng.random() < 0.8}
        order = [w for w in ["w2", "w1", "w3"] if rng.random() < 0.8]
        yield master, workers, order


EMPTY_AUDIO = {"waveform": torch.zeros(1, 2, 1), "sample_rate": 44100}


def reference_audio_combination():
    collector, _, _ = ref_collector.load()
    node = collector.DistributedCollectorNode()
    return [fingerprint(node._combine_audio(master, workers, EMPTY_AUDIO, order)) for master, workers, order in _audio_cases()]


def test_audio_combination_matches_reference():
    """nodes/collector.py:121-174 (the reference's _combine_audio) against our combine_audio on the same piece sets."""
    from __graft_entry__ import load_package
    load_package()
    from comfyui_distributed_b200.nodes.collector import combine_audio
    want = reference_fingerprints("test_collector_vs_reference")["combine_audio"]
    cases = list(_audio_cases())
    assert len(want) == len(cases)
    for (master, workers, order), ref in zip(cases, want):
        seq = [master] + [workers.get(w) for w in order] + [workers[w] for w in sorted(workers) if w not in order]
        got = fingerprint(combine_audio(seq, EMPTY_AUDIO))
        assert got["sample_rate"] == ref["sample_rate"]
        assert got["waveform"] == ref["waveform"]
