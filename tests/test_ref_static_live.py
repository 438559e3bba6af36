"""The REAL reference's multi-worker static mode -- master and workers over aiohttp with its PNG transport,
oracle/ref_static_run.py -- and `oracle.replay_static` of the tile assignment that run's pull queue produced agree
bit for bit.  The assignment and the result of each run are stored in tests/golden/reference_fingerprints.json;
reference_static_run runs the reference again where its tree is loadable (oracle/gen_reference_fingerprints.py)."""
import numpy as np
import pytest

import ref_static_run
import usdu_oracle as orc
from inputs import fingerprint, make_input, reference_fingerprints

CASES = [(2, 1, 520, 700, 256, 32, 8, True), (1, 5, 200, 260, 128, 16, 4, False)]


def reference_static_run(n_workers, B, H, W, tile, pad, blur, uniform):
    img = make_input("noise", 17, B, H, W)
    res, asg = ref_static_run.run_static(img, n_workers, tile, pad, blur, uniform, 5, 0.5, master_delay=0.1)
    ref = orc.replay_static(img, orc.make_t0_denoiser(5, 0.5), tile, tile, pad, blur, uniform, asg)
    assert np.array_equal(ref, res), asg
    return {"assignment": [list(map(int, a)) for a in asg], "result": fingerprint(res)}


@pytest.mark.parametrize("n_workers,B,H,W,tile,pad,blur,uniform", CASES)
def test_real_static_mode_equals_replay(n_workers, B, H, W, tile, pad, blur, uniform):
    run = reference_fingerprints("test_ref_static_live")["static_run"][repr((n_workers, B, H, W, tile, pad, blur, uniform))]
    asg = run["assignment"]
    assert len(asg) == n_workers + 1
    assert sorted(t for a in asg for t in a) == list(range(len(orc.make_plan(W, H, tile, tile, pad, uniform)[2])))
    img = make_input("noise", 17, B, H, W)
    ref = orc.replay_static(img, orc.make_t0_denoiser(5, 0.5), tile, tile, pad, blur, uniform, asg)
    assert fingerprint(ref) == run["result"], asg
