"""CUDA path (through the C ABI) against outputs of the REFERENCE'S OWN SOURCES (tests/golden/ref_vectors.*.npz, produced by
oracle/_ref/libref.so: /root/reference/src/*.cpp compiled unmodified, see tests/golden/make_ref_vectors.py and tests/test_ref_pin.py).
Bars: flags, match pixels, FAST corners and hypothesis counts bit-exact; x and P within 1e-9 relative."""
import numpy as np
import pytest

from oracle import ref_py as R
from tests import helpers as H
from tests import ref_cases as RC

pytestmark = pytest.mark.gpu


def test_cuda_reproduces_reference_on_bundled_sequence():
    """whole System::TrackRunning loop (map management incl. FAST initialisation and the run-ahead delete, prediction, patch warp,
    ZNCC search, 1-point RANSAC, li / hi updates) over frames of the reference's bundled sequence"""
    assert RC.run_bundled(RC.GpuEngine) == 9


def test_cuda_reproduces_reference_ransac_and_updates():
    RC.run_q1(RC.GpuEngine)


def test_cuda_reproduces_reference_cartesian_conversion():
    RC.run_convert(RC.GpuEngine)


@pytest.mark.skipif(not R.available(), reason="oracle/_ref/libref.so did not travel")
@pytest.mark.parametrize("seed", [41, 42])
def test_cuda_matches_live_reference_on_fresh_inputs(seed):
    N = 30 + seed % 7
    cam, x, P, z, ic = H.q1_consistent_state(N, seed=seed, outlier_frac=0.25)
    r = R.ReferenceFilter()
    e = RC.GpuEngine(r.camera9(), N)
    e.load_map(x, P, z)
    for i in range(N):
        r.add_feature(0, None, None, np.zeros(3), np.eye(3), z[i])
    r.set_state(x, P, prior=True)
    r.set_state(x, P, prior=False)
    e.search(None)
    r.predict_only()
    fr = r.features()
    assert np.array_equal(e.features()["has_h"], fr["has_h"])
    e.set_matches(z, ic & fr["has_h"])
    r.set_matches(z, ic & fr["has_h"])
    dr = R.make_draws(np.random.default_rng(seed), 1000)
    r.set_draws(dr)
    r.ransac_hypotheses()
    rc, run = e.ransac(R.draws_to_u01(dr))
    assert rc == 0 and run == r.draws_consumed()
    assert np.array_equal(e.features()["li"], r.features()["li"])
    for stage in ("update_li", "rescue_hi", "update_hi"):
        getattr(e, stage)()
        getattr(r, stage)()
        xg, Pg = e.state()
        xr, Pr = r.get_state()
        H.assert_x_close(xg, xr, what=f"x after {stage}")
        H.assert_P_close(Pg, Pr, what=f"P after {stage}")
        assert np.array_equal(e.features()["hi"], r.features()["hi"])
