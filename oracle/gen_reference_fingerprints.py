"""Generate tests/golden/reference_fingerprints.json by RUNNING THE REAL REFERENCE (its tree at
$USDU_REFERENCE_ROOT, or where oracle/ref_loader.py finds it).

    python oracle/gen_reference_fingerprints.py

The side-by-side tests (test_conditioning, test_model_patch, test_comfy_sampler_vs_reference,
test_collector_vs_reference, test_ref_static_live) each hold a reference_* function that computes the reference's
side of the comparison on the test's own inputs; this script calls them for every case and stores the results as
tests/inputs.fingerprint (shapes, dtypes and SHA-256 of every tensor), which the tests compare our side against.
Test infrastructure only (see oracle/usdu_oracle.py header).
"""
from __future__ import annotations

import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
TESTS = os.path.join(ROOT, "tests")
for p in (ROOT, HERE, TESTS):
    if p not in sys.path:
        sys.path.insert(0, p)


def main() -> int:
    import ref_collector
    import ref_loader
    if not (ref_loader.available() and ref_collector.available()):
        raise SystemExit(f"reference tree not found at {ref_loader.REF_ROOT}")
    import test_collector_vs_reference as t_col
    import test_comfy_sampler_vs_reference as t_smp
    import test_conditioning as t_cond
    import test_model_patch as t_mp
    import test_ref_static_live as t_static

    out = {
        "test_conditioning": {
            "control_hint_crop": {t_cond._key(*c): t_cond.reference_control_hint_crop(*c) for c in t_cond.REGIONS},
            "area_gligen_reflatents": {t_cond._key(*c): t_cond.reference_area_gligen_reflatents(*c) for c in t_cond.REGIONS},
        },
        "test_model_patch": {
            "crop_model_cond": {repr((lc, region, canvas)): t_mp.reference_crop_model_cond(lc, region, canvas)
                                for lc in (False, True)
                                for region, canvas in ((t_mp.REGION, t_mp.CANVAS), ((0, 0, 544, 544), (1300, 1100)),
                                                       ((724, 524, 1300, 1100), (1300, 1100)))},
        },
        "test_comfy_sampler_vs_reference": {
            "process_tiles_batch": {t_smp._key(*c, *td): t_smp.reference_process_tiles_batch(*c, *td)
                                    for c in t_smp.CASES for td in t_smp.TILED},
        },
        "test_collector_vs_reference": {"combine_audio": t_col.reference_audio_combination()},
        "test_ref_static_live": {"static_run": {repr(c): t_static.reference_static_run(*c) for c in t_static.CASES}},
    }
    path = os.path.join(TESTS, "golden", "reference_fingerprints.json")
    with open(path, "w") as f:
        json.dump({"generator": "oracle/gen_reference_fingerprints.py", "reference": "a91f9fb", "tests": out}, f,
                  separators=(",", ":"))
        f.write("\n")
    print(f"wrote {path} ({os.path.getsize(path)} bytes)")
    return 0


if __name__ == "__main__":
    sys.exit(main())
