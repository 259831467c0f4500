"""Pins the CPU oracle to the REFERENCE'S OWN SOURCES.

tests/golden/ref_vectors.*.npz holds outputs of /root/reference/src/{ExtendKF,Tracking,Converter,Map}.cpp, compiled unmodified
(oracle/Makefile `ref`, stand-in Eigen / OpenCV / ROS headers in oracle/ref_shim/) and driven through the reference's own
TrackRunning call sequence.  The oracle must reproduce them: flags, match pixels and hypothesis counts exactly, x and P to 1e-9.
Where oracle/_ref/libref.so is present (the build container; the GPU box when the prebuilt library travelled) the live library is
checked too: it must regenerate the committed vectors bit for bit, and agree with the oracle on fresh random inputs."""
import os

import numpy as np
import pytest

from oracle import oracle_py as O
from oracle import ref_py as R
from tests import helpers as H
from tests import ref_cases as RC

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_ref = pytest.mark.skipif(not R.available(), reason="oracle/_ref/libref.so not built (needs /root/reference)")


def test_oracle_reproduces_reference_on_bundled_sequence():
    assert RC.run_bundled(RC.OracleEngine) == 9


def test_oracle_sparse_mode_reproduces_reference_on_bundled_sequence():
    assert RC.run_bundled(lambda cam9, n: RC.OracleEngine(cam9, n, dense=False), frames=4) == 4


def test_oracle_reproduces_reference_ransac_and_updates():
    RC.run_q1(RC.OracleEngine)


def test_oracle_reproduces_reference_cartesian_conversion():
    RC.run_convert(RC.OracleEngine)


def test_reference_build_recipe_compiles_the_sources_where_they_lie():
    """no copy of the reference's sources in this repository: the recipe names them under $(REF)/src"""
    mk = open(os.path.join(ROOT, "oracle", "Makefile")).read()
    assert "REF ?= /root/reference" in mk and "$(REF)/src/%.cpp" in mk and "--wrap=rand" in mk
    for dp, _, files in os.walk(ROOT):
        if ".git" in dp or "gpurun_out" in dp:
            continue
        for fn in files:
            assert fn not in ("Tracking.cpp", "ExtendKF.cpp", "Converter.cpp", "Map.cpp", "System.cpp"), os.path.join(dp, fn)
    gi = open(os.path.join(ROOT, ".gitignore")).read()
    assert "oracle/_ref/" in gi
    if os.path.exists(os.path.join(ROOT, ".gpurunignore")):
        assert "oracle/_ref" not in open(os.path.join(ROOT, ".gpurunignore")).read()


@needs_ref
def test_live_reference_regenerates_the_committed_vectors():
    g = RC.load()
    frames = np.load(os.path.join(RC.GOLD, "pgm_frames.npz"))["frames"]
    r = R.ReferenceFilter()
    assert np.array_equal(r.camera9(), g["camera9"])
    for k in range(3):
        pre = f"bundled_k{k}_"
        r.set_draws(np.concatenate([g[pre + "draws_map"][: int(g[pre + "used"][0])], g[pre + "draws_ransac"]]))
        r.track_running(frames[k])  # the whole frame in one call, one rand queue: exactly System::TrackRunning
        assert r.draws_consumed() == int(g[pre + "used"].sum()) and r.draws_underflow() == 0
        x, P = r.get_state()
        assert np.array_equal(x, g[pre + "x"]) and np.array_equal(P, g[pre + "P"])
        f = r.features()
        assert np.array_equal(f["hi"], g[pre + "hi"]) and np.array_equal(f["li"], g[pre + "li"])


@needs_ref
@pytest.mark.parametrize("seed", [31, 32, 33])
def test_oracle_matches_live_reference_on_fresh_inputs(seed):
    N = 14 + seed % 5
    cam, x, P, z, ic = H.q1_consistent_state(N, seed=seed, outlier_frac=0.3)
    r = R.ReferenceFilter()
    o = O.OracleFilter(r.camera9())
    o.set_options(O.Q_ALL, sparse=False, fast_corr=False, warp_patches=True)
    for i in range(N):
        o.add_feature(0, None, np.zeros((13, 13)), np.zeros(3), np.eye(3), z[i])
        r.add_feature(0, None, None, np.zeros(3), np.eye(3), z[i])
    for prior in (True, False):
        o.set_state(x, P, prior=prior)
        r.set_state(x, P, prior=prior)
    o.search_ic_matches(None)
    r.predict_only()
    fo, fr = o.features(), r.features()
    assert np.array_equal(fo["has_h"], fr["has_h"])
    np.testing.assert_allclose(fo["h"], fr["h"], rtol=1e-13, atol=1e-11)
    np.testing.assert_allclose(fo["S"], fr["S"], rtol=1e-10, atol=1e-13)
    for i in range(0, N, 5):  # dense Jacobians, entry by entry
        np.testing.assert_allclose(o.H_dense(i), r.H_dense(i), rtol=1e-11, atol=1e-12)
    o.set_matches(z, ic & fo["has_h"])
    r.set_matches(z, ic & fr["has_h"])
    dr = R.make_draws(np.random.default_rng(seed), 1000)
    r.set_draws(dr)
    r.ransac_hypotheses()
    rc, info = o.ransac_hypotheses(R.draws_to_u01(dr))
    assert rc == 0 and info["hyp_run"] == r.draws_consumed()
    assert np.array_equal(o.features()["li"], r.features()["li"])
    for stage in ("update_li", "rescue_hi", "update_hi"):
        getattr(o, stage)()
        getattr(r, stage)()
        xo, Po = o.get_state()
        xr, Pr = r.get_state()
        H.assert_x_close(xo, xr, what=f"x after {stage}")
        H.assert_P_close(Po, Pr, what=f"P after {stage}")
        assert np.array_equal(o.features()["hi"], r.features()["hi"])


@needs_ref
def test_distortion_model_matches_live_reference():
    r = R.ReferenceFilter()
    o = O.OracleFilter(r.camera9())
    uv = np.random.default_rng(4).uniform([0, 0], [320, 240], (200, 2))
    assert np.array_equal(o.distort(uv), r.distort(uv))
    assert np.array_equal(o.undistort(uv), r.undistort(uv))


# ---- the stand-in third-party headers themselves (oracle/ref_shim/, through oracle/shim_probe.cpp) --------------------------------------
def test_shim_opencv_primitives_match_cv2_fixtures():
    """mini_cv.h's remap / calcCovarMatrix / FAST against cv2 4.13 outputs"""
    import ctypes as C

    L = O.shim_lib()
    fx = np.load(os.path.join(RC.GOLD, "cv_fixtures.npz"))
    for k in range(6):
        src = np.ascontiguousarray(fx[f"remap_src_{k}"], np.float32)
        mx = np.ascontiguousarray(fx[f"remap_mx_{k}"], np.float32)
        my = np.ascontiguousarray(fx[f"remap_my_{k}"], np.float32)
        out = np.zeros(mx.shape, np.float32)
        L.ref_cv_remap(src.ctypes.data_as(C.c_void_p), C.c_int(src.shape[0]), C.c_int(src.shape[1]), mx.ctypes.data_as(C.c_void_p), my.ctypes.data_as(C.c_void_p),
                       C.c_int(mx.shape[0]), C.c_int(mx.shape[1]), out.ctypes.data_as(C.c_void_p))
        assert np.array_equal(out, fx[f"remap_dst_{k}"]), k
    for k in range(3):
        M = np.ascontiguousarray(fx[f"covar_M_{k}"], np.float32)
        cov = fx[f"covar_cov_{k}"]
        got = np.zeros((M.shape[1], M.shape[1]))
        L.ref_cv_calc_covar(M.ctypes.data_as(C.c_void_p), C.c_int(M.shape[0]), C.c_int(M.shape[1]), got.ctypes.data_as(C.c_void_p))
        scale = np.sqrt(np.outer(np.diag(cov), np.diag(cov)))  # the correlation matrix Converter::corrcoef_opencv makes of it
        np.testing.assert_allclose(got / scale, cov / scale, rtol=0, atol=5e-15)
    ff = np.load(os.path.join(RC.GOLD, "fast_fixtures.npz"))
    total = 0
    for name in ff["names"]:
        img = np.ascontiguousarray(ff[f"{name}_img"], np.uint8)
        for t in (100, 40):
            want = ff[f"{name}_kp{t}"]
            xy = np.zeros((20000, 2), np.int32)
            n = L.ref_cv_fast(img.ctypes.data_as(C.c_void_p), C.c_int(img.shape[0]), C.c_int(img.shape[1]), C.c_int(t), C.c_int(1), C.c_int(20000),
                              xy.ctypes.data_as(C.c_void_p))
            assert n == len(want) and np.array_equal(xy[:n], want), (name, t)
            total += n
    assert total > 300


def test_shim_eigen_semantics_match_numpy():
    """the Eigen behaviours the reference's sources rely on, as mini_eigen.h implements them, against numpy (oracle/shim_probe.cpp:
    ref_eigen_probe lists them; the first is the row-by-row comma initialiser behind quirk Q16)"""
    import ctypes as C

    L = O.shim_lib()
    n = 6
    rng = np.random.default_rng(12)
    A = np.asfortranarray(rng.uniform(0.1, 1.0, (n, n)) + 2.0 * np.eye(n))
    v = rng.uniform(-1, 1, n)
    out = np.zeros(4096)
    cnt = L.ref_eigen_probe(A.ctypes.data_as(C.c_void_p), v.ctypes.data_as(C.c_void_p), C.c_int(n), out.ctypes.data_as(C.c_void_p), C.c_int(out.size))
    assert cnt > 0
    pos = [0]

    def take(r, c):
        m = out[pos[0]:pos[0] + r * c].reshape((r, c), order="F")
        pos[0] += r * c
        return m

    assert np.array_equal(take(3, 2), np.array([[1, 2], [3, 4], [5, 6]]))  # row by row
    assert np.array_equal(take(n, n), A)  # four blocks reassemble the matrix
    assert np.array_equal(take(n + 2, 1)[:, 0], np.concatenate([v[:2], [7.0], v[2:], [9.0]]))
    np.testing.assert_allclose(take(n, n), np.linalg.inv(A), rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(take(3, 3), np.linalg.inv(A[:3, :3]), rtol=1e-13, atol=1e-15)
    np.testing.assert_allclose(take(2, 2), np.linalg.inv(A[1:3, 1:3]), rtol=1e-13, atol=1e-15)
    B = A.copy()
    B[1:3, 1:3] = 5.0 * np.eye(2)
    B[0:2, 0] = [-1, -2]
    B[2, 3] = 42.0
    assert np.array_equal(take(n, n), B)
    assert np.array_equal(take(1, n)[0], v) and np.array_equal(take(n, 1)[:, 0], v)
    ru = np.sqrt(A[0] ** 2 + A[1] ** 2)
    np.testing.assert_allclose(take(1, n)[0], ru / (1 + 0.06333 * ru**2 + 0.0139 * ru**4), rtol=1e-15)
    np.testing.assert_allclose(take(1, 1)[0, 0], v @ A @ v, rtol=1e-14)
    np.testing.assert_allclose(take(n, n), A @ np.diag(v), rtol=1e-15)
    assert list(take(4, 1)[:, 0][:2]) == [7.0, 1.0]  # first maximum
    pos[0] -= 2
    nan_max, nan_idx = take(2, 1)[:, 0]
    assert np.isnan(nan_max) and nan_idx == 0  # sticky NaN of slot 0
    S2 = A[:2, :2] @ A[:2, :2].T
    np.testing.assert_allclose(take(2, 1)[:, 0], np.linalg.eigvalsh(S2), rtol=1e-13)
    assert np.array_equal(take(n * n // 2, 2), A.reshape((n * n // 2, 2), order="F"))
    assert np.array_equal(take(n * n, 1)[:, 0], A.reshape(-1, order="F"))
    assert np.array_equal(take(n, 1)[:, 0], (A < 0.5).sum(axis=1))
    np.testing.assert_allclose(take(3, 1)[:, 0], np.cross(v[:3], v[2:5]), rtol=1e-15, atol=1e-17)
    np.testing.assert_allclose(take(1, 1)[0, 0], np.linalg.norm(v), rtol=1e-15)
    assert np.array_equal(take(1, 3)[0], v[1:4])
    assert pos[0] == cnt
