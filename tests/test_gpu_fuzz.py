"""A fixed slice of tools/fuzz_parity.py: random small scenes (map sizes 1 .. 70, every combination of the quirk switches) and, from case
10000 on, maps of 100 .. 300 features (the large-path update from N = 129, multi-CTA rescue), three frames each through rslam_frame (every third case with the patch warp on), against the CPU oracle (dense and sparse mode alternate): match / inlier sets, RANSAC replay counters bit for
bit, x and P to 1e-9, P exactly symmetric."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import fuzz_parity  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("first", [0, 8, 16, 10000])
def test_random_small_scenes_against_the_oracle(first):
    seen = set()
    for case in range(first, first + 8):
        fuzz_parity.run_case(case)
        seen.add(fuzz_parity.case_params(case)["N"])
    assert len(seen) >= 3  # the slice covers several map sizes
