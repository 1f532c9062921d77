#!/usr/bin/env python
"""Generates tests/golden/tracker_golden.npz: the scenarios of tests/tracker_cases.py run through the lifecycle
steps with the REAL cv2 4.13 operators (calcOpticalFlowPyrLK, goodFeaturesToTrack, circle, cvtColor) and the
reference's own of_library.static_immobile / of_library.r_tilde / solve_lgs (AST-extracted from the checkout that
OFB_REFERENCE_DIR names). Also stores cv2.circle masks for a set of radii / centres (the exclusion mask of
velocity_measurment_node:159-161).

Generates tests/golden/tracker_random_golden.npz: the random sequences of tracker_cases.random_case through the
same cv2 operators, with the reference's three functions where the reference is available and otherwise with the
oracle's pinned restatements of them; the file's `arithmetic` entry records which."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
import tracker_cases as tc  # noqa: E402
from oracle import ref_loader, tracker_oracle  # noqa: E402


def random_golden():
    import cv2
    assert cv2.__version__.startswith("4.13"), cv2.__version__
    reference = ref_loader.available()
    eng = tc.cv2_engine(reference=reference)
    g = {"arithmetic": np.array("reference" if reference else "oracle")}
    for seed in tc.RANDOM_SEEDS:
        frames, imus, kw = tc.random_case(seed)
        res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **kw), frames, imus)
        for k, v in tc.pack(res, kw["max_features"] + kw["min_features"]).items():
            g["s%d_%s" % (seed, k)] = v
        print("seed", seed, "n_points", g["s%d_n_points" % seed].tolist(), "added", g["s%d_n_added" % seed].tolist())
    out = os.path.join(ROOT, "tests", "golden", "tracker_random_golden.npz")
    np.savez_compressed(out, **g)
    print("wrote", out, os.path.getsize(out), "bytes, arithmetic:", g["arithmetic"])


def main():
    import cv2
    random_golden()
    if not ref_loader.available():
        sys.exit("tracker_golden.npz not rewritten: " + ref_loader.MISSING)
    eng = tc.cv2_engine()
    g = {}
    for name in tc.SCENARIOS:
        frames, imus, kw = tc.build(name)
        res = tc.run_oracle_tracker(lambda: tracker_oracle.TrackerOracle(tc.W, tc.H, engine=eng, **kw), frames, imus)
        cap = kw["max_features"] + kw["min_features"]
        for k, v in tc.pack(res, cap).items():
            g["%s_%s" % (name, k)] = v
        print(name, "n_points", g[name + "_n_points"].tolist(), "added", g[name + "_n_added"].tolist(),
              "kept", g[name + "_n_kept"].tolist(), "tracked", g[name + "_n_tracked"].tolist())
    # cv2.circle masks: radii x centres incl. partly / fully outside the image
    rng = np.random.default_rng(77)
    masks, meta = [], []
    for radius in (0, 1, 2, 3, 5, 8, 13, 30, 47):
        pts = np.concatenate([rng.uniform(-20, 120, (6, 2)), [[0, 0], [99.9, 63.2], [-radius, 10], [50, 64 + radius]]])
        m = np.ones((64, 100), np.uint8)
        for x, y in pts:
            cv2.circle(m, (int(x), int(y)), radius, 0, cv2.FILLED)
        masks.append(m)
        meta.append(np.concatenate([[radius], pts.reshape(-1)]))
    g["circle_masks"] = np.stack(masks)
    g["circle_meta"] = np.stack(meta)
    out = os.path.join(ROOT, "tests", "golden", "tracker_golden.npz")
    np.savez_compressed(out, **g)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
