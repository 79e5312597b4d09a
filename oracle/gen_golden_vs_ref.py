#!/usr/bin/env python
"""oracle/gen_golden_vs_ref.py — TEST INFRASTRUCTURE ONLY.  Writes tests/golden/vs_ref/<case>.npz: the records the
scenarios of tests/test_oracle_vs_ref.py take from the REFERENCE'S OWN sources (oracle/_ref/libref_f{32,64}.so,
built by oracle/build_ref.py from the reference tree named by EKF_REFERENCE_ROOT).  The test replays each scenario
on the oracle and compares with these files."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import ekfb200  # noqa: E402
import refbind  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402


def main():
    pkg = ekfb200.load_package()
    refbind.build()
    out = os.path.join(ROOT, "tests", "golden", "vs_ref")
    os.makedirs(out, exist_ok=True)

    def save(case, rec):
        path = os.path.join(out, case + ".npz")
        T.save_record(path, rec)
        print(f"{case}: {os.path.getsize(path) / 1024:.0f} KiB")

    for fp64 in (True, False):
        def make(cfg):
            return refbind.ReferenceFilter(cfg, fp64=fp64)
        for params in T.SEQUENCES:
            save(T.case_id("sequence", fp64, *params), T.run_sequence(pkg, make, *params)[0])
        save(T.case_id("controls", fp64), T.run_controls_remove_and_accessors(pkg, make)[0])
        save(T.case_id("xyz", fp64), T.run_xyz_conversion(pkg, make)[0])
        save(T.case_id("blur", fp64), T.run_motion_blur_templates(pkg, make)[0])
        save(T.case_id("forse_plane", fp64), T.run_forse_plane(pkg, make)[0])
        for params in T.RTS_CASES:
            save(T.case_id("rts", fp64, *params), T.run_rts_epoch(pkg, make, *params)[0])
        save(T.case_id("deleted", fp64), T.run_deleted_archive(pkg, make)[0])
    frames, tm, h, S = T.find_match_inputs(pkg)
    uv = np.array([refbind.find_match(frames[0], tm[k], h[k], S[k], sigma_size=3.0, fp64=False) for k in range(len(tm))],
                  dtype=np.int32)
    save(T.case_id("find_match", False), {"uv": uv})


if __name__ == "__main__":
    main()
