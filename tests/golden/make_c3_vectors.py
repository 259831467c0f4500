"""Writes tests/golden/c3_vectors.*.npz: outputs of the CPU oracle (sparse mode) for one whole frame of configuration C3 (N = 2000, state
dimension 12013), with the reference's quirks on (Q1: one low-innovation inlier, ~1990 rescued high-innovation inliers, k ~ 3980) and
with Q1 off (a real low-innovation set).  ~3 minutes per case on 8 cores.  Run from the repository root:
    python tests/golden/make_c3_vectors.py"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import c3_case as C3  # noqa: E402
from tests import golden_npz  # noqa: E402

if __name__ == "__main__":
    cam, scene, seq, P0 = C3.inputs()
    out = dict(digest=np.array(C3.input_digest(scene, seq, P0)))
    for tag, quirks in (("q1on", 0x7), ("q1off", 0x6)):
        t0 = time.time()
        r = C3.run_oracle(quirks, cam, scene, seq, P0)
        print(tag, "info", r["info"], "ic/li/hi", r["ic"].sum(), r["li"].sum(), r["hi"].sum(), f"{time.time() - t0:.0f} s", flush=True)
        for k, v in r.items():
            out[f"{tag}_{k}"] = v
    golden_npz.save("c3_vectors", out)
