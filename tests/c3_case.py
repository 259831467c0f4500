"""The full-size configuration C3 (N = 2000 features, state dimension 12013, P = 1.15 GB) as a deterministic test case: inputs built
with element-wise numpy only, so that the committed outputs of the CPU oracle (tests/golden/c3_vectors.*.npz, written by
tests/golden/make_c3_vectors.py) belong to exactly the inputs the GPU test rebuilds on the box."""
import hashlib

import numpy as np

from ransac_slam_b200 import synth

N = 2000
N_U01 = 16384
STD_SCALE = 0.25
SAMPLES = 100000


def inputs():
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=STD_SCALE)
    seq = synth.make_sequence(scene, T=1, seed=1235, n_u01=N_U01)
    P0 = synth.assemble_P_numpy(scene)
    return cam, scene, seq, P0


def input_digest(scene, seq, P0):
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(scene.x0).tobytes())
    h.update(np.ascontiguousarray(seq.images[0]).tobytes())
    h.update(np.ascontiguousarray(seq.u01[0]).tobytes())
    h.update(np.ascontiguousarray(P0[:, ::97]).tobytes())
    h.update(np.ascontiguousarray(np.diag(P0)).tobytes())
    return h.hexdigest()


def probes(n):
    """where the covariance is compared: the diagonal, SAMPLES random entries and three random projections P v"""
    rng = np.random.default_rng(20261018)
    ii = rng.integers(0, n, SAMPLES)
    jj = rng.integers(0, n, SAMPLES)
    V = rng.standard_normal((n, 3))
    return ii, jj, V


def summarize(x, P):
    ii, jj, V = probes(x.size)
    return dict(x=x.copy(), diag=np.diag(P).copy(), samples=P[ii, jj].copy(), PV=P @ V, absPV=np.abs(P) @ np.abs(V), maxdiag=float(np.abs(np.diag(P)).max()))


def assert_summary_close(got, exp, what, rtol=1e-9):
    """x, P to the north-star bar: |d| <= rtol * max(|a|, |b|) + 1e-12 * max diag P (DESIGN.md section 4)"""
    atol = 1e-12 * float(exp["maxdiag"])
    for key in ("diag", "samples"):
        a, b = got[key], exp[key]
        d = np.abs(a - b)
        lim = rtol * np.maximum(np.abs(a), np.abs(b)) + atol
        assert (d <= lim).all(), f"{what}: P {key}: {(d > lim).sum()} entries off, max |d| = {d.max():.3e}"
    # projections: every entry of P enters; the bound is the entrywise bar summed along each row
    d = np.abs(got["PV"] - exp["PV"])
    lim = rtol * exp["absPV"] + atol * np.sqrt(got["x"].size)
    assert (d <= lim).all(), f"{what}: P v: max |d| / bound = {(d / lim).max():.3e}"
    # state: 1e-9 relative, with an absolute floor of 1e-10 (metres / radians / inverse metres) for entries that are themselves ~0 --
    # two chained updates of rank ~2000 leave ~2e-11 of absolute difference between a Cholesky-based and an LU-based solve
    a, b = got["x"], exp["x"]
    d = np.abs(a - b)
    assert (d <= rtol * np.maximum(np.abs(a), np.abs(b)) + 1e-10).all(), f"{what}: x: max |d| = {d.max():.3e} at {int(np.argmax(d))}"


def run_oracle(quirks, cam, scene, seq, P0, threads=None):
    """one whole frame of the CPU oracle in sparse mode (structural zeros skipped, same formulas); returns the fixture dict"""
    import os

    from oracle import oracle_py as O

    O.set_threads(threads or os.cpu_count() or 1)
    o = O.OracleFilter(cam.as9(), std_a=0.007 * STD_SCALE, std_alpha=0.007 * STD_SCALE, std_z=scene.std_z, quirks=quirks, sparse=True, fast_corr=True,
                       warp_patches=False)
    for i in range(N):
        o.add_feature(0, None, scene.templates[i].astype(np.float64), scene.x0[:3], np.eye(3), scene.uv0[i])
    o.set_state(scene.x0, P0)
    o.map_reset_flags()
    o.ekf_prediction()
    o.search_ic_matches(seq.images[0])
    rc, info = o.ransac_hypotheses(seq.u01[0])
    out = dict(info=np.array([rc, info["hyp_run"], info["best_support"], info["n_hyp"], info["num_ic"]]))
    o.update_li()
    x, P = o.get_state()
    for k, v in summarize(x, P).items():
        out["li_" + k] = v
    del P
    o.rescue_hi()
    o.update_hi()
    f = o.features()
    for k in ("ic", "li", "hi", "has_h", "z", "h"):
        out[k] = f[k]
    x, P = o.get_state()
    for k, v in summarize(x, P).items():
        out["hi_" + k] = v
    return out
