"""The kernels in front of the EKF update -- k_ekf_prediction, k_predict (mode 0: h, H and S for the search; mode 1: the rescue gate)
and k_search (the ZNCC active search) -- against float64 and exact references, at the edges where they can go wrong.

In a whole frame the data decide the map size, the search window, the gates and the image layout, so those edges are reached by
chance.  Here the state is uploaded directly (rslam_upload_state / rslam_upload_linearisation / rslam_set_matches), and the search
inputs h, S, has_h and the predicted patch are written into a snapshot (rslam_checkpoint_save), patched and loaded back, so that
every case controls exactly what the kernel sees.  Each case names the edge it exists for.

References:
- prediction: oracle/np_oracle.py::ekf_prediction (checked against the C++ oracle here), x and P at the project's 1e-9 bar;
- measurement prediction: np_oracle.predict_h / jacobian_H and a dense S = H P H^T + I;
- search: an exact ZNCC over integer-valued patches and images.  With 169 pixels, every candidate's centred sums
  169 sum(ab) - sum(a) sum(b), 169 sum(a^2) - sum(a)^2 and 169 sum(b^2) - sum(b)^2 are integers, so scores are compared with each other
  and with corr_threshold in exact arithmetic.  A match must equal the exact arg-max when it is decided (top two scores more than
  1e-12 apart, relative, and the best not within 1e-12 of the threshold).  Identical candidate windows give bitwise identical device
  scores, so the first in the reference's visiting order (x outer, y inner) must win.  Windows tied only in exact arithmetic
  (b and b + c) are decided by rounding in the reference as on the device, so there the match may be any of the tied candidates:
  that band is the only place where the test accepts more than one answer.  The chi-square gate, the eigenvalue gate, the window
  half-widths ceil(2 sqrt(S_ii)) and round(h) are kept at least 1e-12 (relative) from their thresholds, which the CPU tests assert.

The rescue's deferred quaternion normalisation (k_predict with fuse_jnorm) is reachable only through rslam_frame and stays covered by
the frame tests (test_gpu_fuzz, test_gpu_c1, test_gpu_at_size)."""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

from oracle import np_oracle as NP
from ransac_slam_b200 import capi, synth
from tests import helpers as H

CAM9 = synth.Camera().as9()
# the same sensor behind a short lens (f / dx = 50 px): the +-60 degree cone lies inside the image, so the cone alone decides visibility
CAM_WIDE = CAM9.copy()
CAM_WIDE[6] = 0.56
ROWS, COLS = 240, 320
CHI2, CORR_THR, MAX_EIG = 5.9915, 0.80, 100.0
STD_A = STD_ALPHA = 0.007
Q_ALL, Q4, Q6 = 0x7, 0x2, 0x4
T60 = 1.7320508075688772
HP = 6  # half patch


# ---- maps ------------------------------------------------------------------------------------------------------------------------
def layout(types):
    sizes = np.where(np.asarray(types) == 0, 6, 3)
    offs = 13 + np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(int)
    return offs[:len(types)], sizes, 13 + int(sizes.sum())


def spd(n, sd, rng, rank=6, a=0.1):
    """D (a U U^T / r + diag(d)) D: every entry non-zero, SPD, exactly symmetric"""
    U = rng.standard_normal((n, rank)) * np.sqrt(a / rank)
    C = U @ U.T
    C[np.diag_indices(n)] += rng.uniform(0.5, 1.5, n)
    P = C * sd[:, None] * sd[None, :]
    return np.asfortranarray(0.5 * (P + P.T))


def camera_state(rng, w=None):
    x = np.zeros(13)
    x[0:3] = rng.normal(0, 0.05, 3)
    q = np.array([1.0, *rng.normal(0, 0.03, 3)])
    x[3:7] = q / np.linalg.norm(q)
    x[7:10] = rng.normal(0, 0.01, 3)
    x[10:13] = rng.normal(0, 0.01, 3) if w is None else w
    return x


@functools.lru_cache(maxsize=8)
def random_map(N, n_cart=0, seed=0, w=None):
    """A map for the prediction: N features (the last n_cart cartesian), generic x and P.  Returns (types, x, P), read only."""
    rng = np.random.default_rng([N, n_cart, seed, 21])
    types = np.zeros(N, np.int32)
    types[N - n_cart:] = 1
    offs, sizes, n = layout(types)
    x = np.zeros(n)
    x[:13] = camera_state(rng, None if w is None else np.array(w))
    sd = np.full(n, 0.01)
    sd[:13] = [0.004] * 3 + [0.001] * 4 + [0.01] * 3 + [0.003] * 3
    for i in range(N):
        o = offs[i]
        x[o:o + 3] = rng.normal(0, 1, 3)
        if types[i] == 0:
            x[o + 3:o + 6] = rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.4), 1 / rng.uniform(2, 15)
    P = spd(n, sd, rng)
    for v in (types, x, P):
        v.flags.writeable = False
    return types, x, P


def undistort(cam, uv):  # ExtendKF::undistort_fm (src/ExtendKF.cpp:266-285)
    k1, k2, _, _, Cx, Cy, _, dx, dy = cam
    xd, yd = (uv[0] - Cx) * dx, (uv[1] - Cy) * dy
    rd2 = xd * xd + yd * yd
    D = 1 + k1 * rd2 + k2 * rd2 * rd2
    return np.array([xd * D / dx + Cx, yd * D / dy + Cy])


def ray(cam, uv_d, depth):
    """camera-frame point at `depth` whose distorted pixel is uv_d"""
    k1, k2, _, _, Cx, Cy, f, dx, dy = cam
    u, v = undistort(cam, uv_d)
    return np.array([(u - Cx) * dx / f, (v - Cy) * dy / f, 1.0]) * depth


def place(x, types, i, p_cam, rng):
    """write feature i so that its camera-frame point is p_cam (inverse depth: from an anchor near the camera)"""
    offs, _, _ = layout(types)
    o = offs[i]
    t, R = x[0:3], NP.q2r(x[3:7])
    p = t + R @ p_cam
    if types[i] == 1:
        x[o:o + 3] = p
        return
    a = t + rng.normal(0, 0.03, 3)
    d = p - a
    if p_cam[2] < 0:  # behind the camera: keep the anchor behind it too, so that hrl_z = (p - t) rho stays negative
        a = t
        d = p - a
    m = d / np.linalg.norm(d)
    x[o:o + 3] = a
    x[o + 3] = np.arctan2(m[0], m[2])
    x[o + 4] = np.arctan2(-m[1], np.hypot(m[0], m[2]))
    x[o + 5] = 1.0 / np.linalg.norm(d)


def map_sd(types, n):
    offs, sizes, _ = layout(types)
    sd = np.zeros(n)
    sd[:13] = [0.004] * 3 + [0.001] * 4 + [0.01] * 3 + [0.003] * 3
    for i, o in enumerate(offs):
        sd[o:o + sizes[i]] = [0.002] * 3 + [0.001, 0.001, 0.02][:sizes[i] - 3]
    return sd


@functools.lru_cache(maxsize=8)
def visible_map(N, seed=0, cart_every=5, cam_key="std"):
    """N features spread over the image (every cart_every-th cartesian) at depths 2..10.  Returns (cam, types, x, P), read only."""
    cam = CAM9 if cam_key == "std" else CAM_WIDE
    rng = np.random.default_rng([N, seed, cart_every, 22])
    types = np.array([1 if cart_every and i % cart_every == cart_every - 1 else 0 for i in range(N)], np.int32)
    _, _, n = layout(types)
    x = np.zeros(n)
    x[:13] = camera_state(rng)
    for i in range(N):
        uv = np.array([rng.uniform(20, COLS - 20), rng.uniform(20, ROWS - 20)])
        place(x, types, i, ray(cam, uv, rng.uniform(2, 10)), rng)
    P = spd(n, map_sd(types, n), rng)
    for v in (types, x, P):
        v.flags.writeable = False
    return cam, types, x, P


# ---- float64 references of the measurement prediction ---------------------------------------------------------------------------
def dense_H(cam, x, types, i, h_i):
    return NP.jacobian_H(cam, x, types, i, h_i)


def S_of(Hd, P):
    idx = np.flatnonzero(np.any(Hd != 0, axis=0))
    Hs = Hd[:, idx]
    return Hs @ P[np.ix_(idx, idx)] @ Hs.T


def assert_close(a, b, rtol=1e-9, what=""):
    a, b = np.asarray(a, float), np.asarray(b, float)
    atol = 1e-12 * max(np.abs(b).max(), 1.0)
    d = np.abs(a - b)
    bad = d > rtol * np.maximum(np.abs(a), np.abs(b)) + atol
    assert not bad.any(), f"{what}: {bad.sum()} entries differ, max |d| = {d.max():.3e}"


def predict_reference(cam, types, x, P, stale):
    """mode-0 expectations: h, has_h, Hc, Hf, S per feature.  stale: {i: h} of features whose h is set before the call."""
    h, vis = NP.predict_h(cam, x, types)
    offs, sizes, _ = layout(types)
    N = len(types)
    out = dict(vis=vis, has_h=vis.copy(), h=h.copy(), Hc=np.zeros((N, 2, 7)), Hf=np.zeros((N, 2, 6)), S=np.zeros((N, 2, 2)))
    for i, hs in stale.items():
        out["has_h"][i] = True
        if not vis[i]:
            out["h"][i] = hs
    for i in np.flatnonzero(out["has_h"]):
        Hd = dense_H(cam, x, types, i, out["h"][i])
        out["Hc"][i] = Hd[:, :7]
        out["Hf"][i, :, :sizes[i]] = Hd[:, offs[i]:offs[i] + sizes[i]]
        out["S"][i] = S_of(Hd, P) + np.eye(2)
    return out


# ---- 1. ekf_prediction ------------------------------------------------------------------------------------------------------------
PRED_CASES = {"n13": (0, 0), "n127": (19, 0), "n130": (20, 1), "n253": (40, 0), "n259": (41, 0), "N600": (600, 7)}


@pytest.mark.parametrize("w", [None, (1e-11, 1e-11, 1e-11)], ids=["w", "w1e-11"])
@pytest.mark.parametrize("N", [3, 40])
def test_np_ekf_prediction_matches_the_cpp_oracle(N, w):
    """np_oracle.ekf_prediction restates ExtendKF::ekf_prediction independently of the C++ oracle; they agree to 1e-12, also at the
    |omega| = 1e-11 of initialize_x_and_p (src/ExtendKF.cpp:32-54)."""
    from oracle import oracle_py as O

    types, x, P = random_map(N, 1, w=w)
    o = O.OracleFilter(CAM9, std_a=STD_A, std_alpha=STD_ALPHA)
    for t in types:
        o.add_feature(int(t), None, np.zeros((13, 13)), np.zeros(3), np.eye(3), np.zeros(2))
    o.set_state(x, P)
    o.ekf_prediction()
    xo, Po = o.get_state(prior=True)
    xr, Pr = NP.ekf_prediction(x, P, STD_A, STD_ALPHA)
    H.assert_x_close(xr, xo, rtol=1e-12)
    H.assert_P_close(Pr, Po, rtol=1e-12)


def check_prediction(f, b, types, x, P):
    xr, Pr = NP.ekf_prediction(x, P, STD_A, STD_ALPHA)
    xg, _ = f.download_state(b=b, prior=True, want_P=False)
    _, Pg = f.download_state(b=b)
    n = x.size
    assert xg.size == n
    H.assert_x_close(xg[:13], xr[:13], what=f"x_k_km1 camera, filter {b}")
    assert np.array_equal(xg[13:], x[13:]), f"x_k_km1 features, filter {b}"
    assert np.array_equal(Pg, Pg.T), f"P symmetric, filter {b}"
    H.assert_P_close(Pg[:13, :13], Pr[:13, :13], what=f"P_cc, filter {b}")
    if n > 13:
        H.assert_P_close(Pg[:13, 13:], Pr[:13, 13:], what=f"P_cf strip, filter {b}")
    assert np.array_equal(Pg[13:, 13:], P[13:, 13:]), f"P_ff must be untouched, filter {b}"


def past_n_unchanged(f, b, big, small_n):
    """re-declare filter b as the larger map `big` (x only): P outside the small map's n x n block must still be big's P"""
    types, x, P = big
    f.upload_state(x, None, feat_types=types, b=b)
    _, Pg = f.download_state(b=b)
    mask = np.ones(P.shape, bool)
    mask[:small_n, :small_n] = False
    assert np.array_equal(Pg[mask], P[mask]), f"P past n = {small_n} changed, filter {b}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PRED_CASES), ids=list(PRED_CASES))
def test_ekf_prediction(case):
    """n = 13 (no features); n = 127 / 130 and 253 / 259 either side of the 128-row CTA boundary; N = 600 (29 CTAs)."""
    N, n_cart = PRED_CASES[case]
    types, x, P = random_map(N, n_cart)
    f = capi.Filter(CAM9, max(N, 1), std_a=STD_A, std_alpha=STD_ALPHA)
    try:
        f.upload_state(x, P, feat_types=types)
        f.ekf_prediction()
        check_prediction(f, 0, types, x, P)
    finally:
        f.close()


@pytest.mark.gpu
def test_ekf_prediction_small_omega_and_ldp_larger_than_n():
    """|omega| = 1e-11 (initialize_x_and_p's value) on a 130-entry state in a handle sized for 300 features (ldp = 1824): P past n is
    bitwise unchanged."""
    small = random_map(20, 1, w=(1e-11, 1e-11, 1e-11))
    big = random_map(300, 0, seed=3)
    f = capi.Filter(CAM9, 300, std_a=STD_A, std_alpha=STD_ALPHA)
    try:
        f.upload_state(big[1], big[2], feat_types=big[0])
        f.upload_state(small[1], small[2], feat_types=small[0])
        f.ekf_prediction()
        check_prediction(f, 0, *small)
        past_n_unchanged(f, 0, big, small[1].size)
    finally:
        f.close()


@pytest.mark.gpu
def test_ekf_prediction_batch_of_13_beside_1000():
    """One batch: n = 1003 (8 CTAs) beside n = 13, whose CTAs 1..7 exit at once and must leave its P past n alone, and a third
    member of n = 259.  The grid is sized for the largest map."""
    big = random_map(165, 0, seed=1)
    members = [big, random_map(0, 0), random_map(41, 0, seed=2)]
    f = capi.Filter(CAM9, 165, batch=3, std_a=STD_A, std_alpha=STD_ALPHA)
    try:
        for b in range(3):
            f.upload_state(big[1], big[2], feat_types=big[0], b=b)
        for b, m in enumerate(members):
            f.upload_state(m[1], m[2], feat_types=m[0], b=b)
        f.ekf_prediction()
        for b, m in enumerate(members):
            check_prediction(f, b, *m)
        for b in (1, 2):
            past_n_unchanged(f, b, big, members[b][1].size)
    finally:
        f.close()


# ---- 2. predict_measurements (k_predict mode 0) ----------------------------------------------------------------------------------
def edge_map(seed=0):
    """Features placed on the edges of the visibility gates (standard camera: the image border; wide camera: the +-60 degree cone),
    behind the camera, and ordinary ones.  Returns {cam_key: (cam, types, x, P, names, stale)}; stale = {i: h} of features whose h
    is set before the call (a visible one gets a new h; an invisible one keeps its stale h)."""
    out = {}
    eps = 1e-9
    for key, cam in (("std", CAM9), ("wide", CAM_WIDE)):
        rng = np.random.default_rng([seed, 23, 0 if key == "std" else 1])
        names, pts = [], []
        if key == "std":
            m = 1e-6  # px, far above the distort / undistort round trip (~1e-12 px)
            for (u, v), nm in [((m, 120.0), "u>0"), ((-m, 120.0), "u<0"), ((COLS - m, 100.0), "u<nCols"), ((COLS + m, 100.0), "u>nCols"),
                               ((150.0, m), "v>0"), ((150.0, -m), "v<0"), ((170.0, ROWS - m), "v<nRows"), ((170.0, ROWS + m), "v>nRows")]:
                names.append(nm)
                pts.append(ray(cam, np.array([u, v]), rng.uniform(2, 8)))
        else:
            for ax in (0, 1):
                for sgn in (1.0, -1.0):
                    for side, s in (("in", 1 - eps), ("out", 1 + eps)):
                        z = rng.uniform(2, 8)
                        p = np.array([0.0, 0.0, z])
                        p[ax] = sgn * T60 * z * s
                        p[1 - ax] = 0.1 * z * rng.uniform(-1, 1)
                        names.append(f"cone{'xy'[ax]}{'+-'[sgn < 0]}-{side}")
                        pts.append(p)
        for k in range(3):
            names.append(f"behind{k}")
            pts.append(np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), -rng.uniform(1, 5)]))
        for k in range(6):
            names.append(f"plain{k}")
            r = 20 if key == "std" else 100  # the wide camera's cone ends inside the image
            pts.append(ray(cam, np.array([rng.uniform(r, COLS - r), rng.uniform(r, ROWS - r)]), rng.uniform(2, 10)))
        N = len(pts)
        types = np.array([(i % 2) for i in range(N)], np.int32)  # both parametrisations at every edge
        _, _, n = layout(types)
        x = np.zeros(n)
        x[:13] = camera_state(rng)
        for i, p in enumerate(pts):
            place(x, types, i, p, rng)
        P = spd(n, map_sd(types, n), rng)
        # stale h: on two invisible features (one behind the camera, one outside the gate) and on one visible feature
        stale = {names.index("behind0"): np.array([100.5, 80.25]), N - 1: np.array([10.0, 20.0])}
        stale[names.index("u<0" if key == "std" else "conex+-out")] = np.array([3.0, 119.0])
        out[key] = (cam, types, x, P, names, stale)
    return out


def test_edge_map_exercises_every_gate():
    """The reference sees each placed feature on its intended side of its gate, so the GPU case tests the gate, not the data."""
    for key, (cam, types, x, P, names, stale) in edge_map().items():
        _, vis = NP.predict_h(cam, x, types)
        for nm, v in zip(names, vis):
            want = not (nm.endswith("out") or nm.startswith("behind") or nm in ("u<0", "u>nCols", "v<0", "v>nRows"))
            assert v == want, (key, nm)


def run_predict(f, b, cam, types, x, P, stale):
    f.upload_state(x, P, feat_types=types, b=b, prior=True)
    N = len(types)
    if stale:
        h0 = np.zeros((N, 2))
        fl = np.zeros((N, 4), np.uint8)
        for i, hs in stale.items():
            h0[i] = hs
            fl[i, 0] = 1
        f.upload_linearisation(h0, None, None, None, fl, b=b)
    return predict_reference(cam, types, x, P, stale)


def check_predict(f, b, ref, stale, what=""):
    fg = f.features(b)
    Hc, Hf = f.H_sparse(b)
    assert np.array_equal(fg["has_h"], ref["has_h"]), what
    hv = ref["has_h"]
    vis = ref["vis"]
    assert_close(fg["h"][vis], ref["h"][vis], what="h " + what)
    for i, hs in stale.items():
        if not vis[i]:
            assert np.array_equal(fg["h"][i], hs), f"stale h of feature {i} {what}"
    assert_close(Hc[hv], ref["Hc"][hv], what="Hc " + what)
    assert_close(Hf[hv], ref["Hf"][hv], what="Hf " + what)
    assert_close(fg["S"][hv], ref["S"][hv], what="S " + what)


@pytest.mark.gpu
@pytest.mark.parametrize("key", ["std", "wide"])
def test_predict_gates_stale_h_and_cartesian(key):
    """Image border (standard camera) and +-60 degree cone (wide camera) at a margin of 1e-6 px / 1e-9 relative on both sides,
    features behind the camera, both parametrisations at every edge, and stale h: a feature that was visible and has left the view
    keeps its h, gets its Jacobian at that h and gets its S (src/ExtendKF.cpp:77-78)."""
    cam, types, x, P, names, stale = edge_map()[key]
    f = capi.Filter(cam, len(types))
    try:
        ref = run_predict(f, 0, cam, types, x, P, stale)
        f.predict_measurements()
        check_predict(f, 0, ref, stale, key)
    finally:
        f.close()


def on_cone_map():
    """Identity pose, cartesian features exactly on the +-60 degree cone (|x| = tan(60 deg) z with z = 4, so the device's hrl and
    tan(60 deg) z are exact) and one 1 ulp outside, wide camera.  The reference's atan2 puts the equality inside (59.99999999999999
    degrees), as the kernel's |x| <= tan(60 deg) z does."""
    pts = []
    for ax in (0, 1):
        for sgn in (1.0, -1.0):
            p = np.array([0.0, 0.0, 4.0])
            p[ax] = sgn * T60 * 4.0
            pts.append(p)
    p = np.array([np.nextafter(T60 * 4.0, 10.0), 0.0, 4.0])
    pts.append(p)
    types = np.ones(len(pts), np.int32)
    x = np.zeros(13 + 3 * len(pts))
    x[3] = 1.0
    for i, q in enumerate(pts):
        x[13 + 3 * i:16 + 3 * i] = q
    P = spd(x.size, map_sd(types, x.size), np.random.default_rng(30))
    return types, x, P


def test_on_cone_map_is_decided_by_the_equality():
    types, x, P = on_cone_map()
    _, vis = NP.predict_h(CAM_WIDE, x, types)
    assert vis.tolist() == [True] * 4 + [False]


@pytest.mark.gpu
def test_predict_exactly_on_the_cone():
    """|x| == tan(60 deg) z bitwise on the device: visible, like the reference; one ulp further out: not visible."""
    types, x, P = on_cone_map()
    f = capi.Filter(CAM_WIDE, len(types))
    try:
        ref = run_predict(f, 0, CAM_WIDE, types, x, P, {})
        f.predict_measurements()
        check_predict(f, 0, ref, {}, "on the cone")
    finally:
        f.close()


@pytest.mark.gpu
@pytest.mark.parametrize("N", [128, 129, 256, 257])
def test_predict_cta_boundaries(N):
    """N = 128 / 129 and 256 / 257 (one thread per feature, 128 per CTA), every fifth feature cartesian."""
    cam, types, x, P = visible_map(N)
    f = capi.Filter(cam, N)
    try:
        ref = run_predict(f, 0, cam, types, x, P, {})
        assert ref["vis"].all()
        f.predict_measurements()
        check_predict(f, 0, ref, {}, f"N = {N}")
    finally:
        f.close()


@pytest.mark.gpu
def test_predict_heterogeneous_batch_ldp_larger_than_n():
    """A batch of 129, 30 and 200 features in a handle sized for 300 (ldp larger than every n); the grid is sized for 200."""
    maps = [visible_map(129, seed=1), visible_map(30, seed=2), visible_map(200, seed=3)]
    f = capi.Filter(CAM9, 300, batch=3)
    try:
        refs = [run_predict(f, b, cam, types, x, P, {}) for b, (cam, types, x, P) in enumerate(maps)]
        f.predict_measurements()
        for b, ref in enumerate(refs):
            check_predict(f, b, ref, {}, f"filter {b}")
    finally:
        f.close()


# ---- 3. rescue_hi (k_predict mode 1) and update_hi ---------------------------------------------------------------------------------
@functools.lru_cache(maxsize=4)
def rescue_case(N, q6):
    """x_k_k = a visible map; every third feature carries a stale h (two of them now out of view); matches z = h + noise on most
    features, some of them low-innovation inliers (skipped by the gate).  Returns the inputs and the reference's hi set, h and H."""
    cam, types, x0, P = visible_map(N, seed=5)
    x = x0.copy()
    rng = np.random.default_rng([N, 24])
    offs, sizes, n = layout(types)
    for i in (3, 6):  # move two features out of view (behind the camera): they keep their stale h
        place(x, types, i, np.array([0.3, 0.2, -2.0]), rng)
    stale = {i: np.array([rng.uniform(30, 290), rng.uniform(30, 210)]) for i in range(0, N, 3)}
    ref = predict_reference(cam, types, x, P, stale)
    ic = ref["has_h"] & (rng.random(N) < 0.9)
    li = ic & (rng.random(N) < 0.15)
    ic[[3, 6]], li[[3, 6]] = True, False  # the two stale-h features are gated
    z = ref["h"] + rng.normal(0, 2.0, (N, 2))
    S = ref["S"] - (np.eye(2) if q6 else 0)
    nu = z - ref["h"]
    chi = np.einsum("ni,nij,nj->n", nu, np.linalg.inv(S), nu)
    need = ic & ~li
    hi = need & (chi < CHI2)
    return dict(cam=cam, types=types, x=x, P=P, stale=stale, ref=ref, ic=ic, li=li, z=z, chi=chi, need=need, hi=hi)


@pytest.mark.parametrize("N", [128, 129])
@pytest.mark.parametrize("q6", [True, False])
def test_rescue_data_stay_off_the_chi2_gate(N, q6):
    """No gated feature's chi-square lies within 1e-9 (relative) of chi2_095_2; both outcomes occur, and stale-h features are gated."""
    c = rescue_case(N, q6)
    g = c["need"]
    assert (np.abs(c["chi"][g] / CHI2 - 1) > 1e-9).all()
    assert 10 < c["hi"].sum() < g.sum() - 5
    assert any(c["need"][i] and not c["ref"]["vis"][i] for i in c["stale"])


@pytest.mark.gpu
@pytest.mark.parametrize("q6", [True, False], ids=["q6", "no-q6"])
@pytest.mark.parametrize("N", [128, 129])
def test_rescue_and_hi_update(N, q6):
    """rslam_rescue_hi at x_k_k against a numpy chi-square gate with quirk Q6 on and off, then rslam_update_hi against
    np_oracle.ekf_update on the reference's hi set.  N = 128: one CTA, the gather is fused into the rescue and update_hi must not
    launch k_upd_gather; N = 129: two CTAs and a separate gather."""
    c = rescue_case(N, q6)
    N_ = len(c["types"])
    f = capi.Filter(c["cam"], N_, quirks=Q_ALL if q6 else Q_ALL & ~Q6)
    try:
        f.upload_state(c["x"], c["P"], feat_types=c["types"])
        h0 = np.zeros((N_, 2))
        fl = np.zeros((N_, 4), np.uint8)
        for i, hs in c["stale"].items():
            h0[i] = hs
            fl[i, 0] = 1
        fl[:, 1] = c["ic"]
        fl[:, 2] = c["li"]
        f.upload_linearisation(h0, None, None, c["z"], fl)
        f.profile(True)
        f.profile_read()
        f.rescue_hi()
        fg = f.features()
        f.update_hi()
        launches = {name: cnt for name, (cnt, _) in f.profile_read().items()}
        f.profile(False)
        assert np.array_equal(fg["hi"], c["hi"])
        assert ("k_upd_gather" in launches) == (N == 129), launches
        assert launches["k_predict"] == 1
        ref = c["ref"]
        idx = np.flatnonzero(c["hi"])
        Hd = np.vstack([dense_H(c["cam"], c["x"], c["types"], i, ref["h"][i]) for i in idx])
        xr, Pr = NP.ekf_update(c["x"], c["P"], Hd, c["z"][idx].reshape(-1), ref["h"][idx].reshape(-1))
        xg, Pg = f.download_state()
        assert np.array_equal(Pg, Pg.T)
        H.assert_x_close(xg, xr)
        H.assert_P_close(Pg, Pr)
    finally:
        f.close()


# ---- 4. match (k_search) -----------------------------------------------------------------------------------------------------------
def c_round(v):  # C round(): half away from zero
    return int(math.floor(v + 0.5)) if v >= 0 else -int(math.floor(-v + 0.5))


def lmax_of(S):
    return 0.5 * (S[0, 0] + S[1, 1]) + math.sqrt(0.25 * (S[0, 0] - S[1, 1]) * (S[0, 0] - S[1, 1]) + S[1, 0] * S[1, 0])


def gate(h, S, cam=CAM9):
    """Tracking::matching's candidate loop (src/Tracking.cpp:295-330): the candidates (j, i) of the box in visiting order (x outer,
    y inner) with their chi-square and whether they pass the chi-square and border tests; margins are asserted, not assumed."""
    nRows, nCols = int(cam[2]), int(cam[3])
    hsx, hsy = math.ceil(2 * math.sqrt(S[0, 0])), math.ceil(2 * math.sqrt(S[1, 1]))
    for v in (2 * math.sqrt(S[0, 0]), 2 * math.sqrt(S[1, 1])):
        assert abs(v - round(v)) > 1e-12 * max(v, 1), "window half-width on an integer"
    for v in h:
        assert abs(v - math.floor(v) - 0.5) > 1e-12 * abs(v), "h on a half-integer"
    cx, cy = c_round(h[0]), c_round(h[1])
    det = S[0, 0] * S[1, 1] - S[0, 1] * S[1, 0]
    out = []
    for j in range(cx - hsx, cx + hsx + 1):
        for i in range(cy - hsy, cy + hsy + 1):
            n0, n1 = j - h[0], i - h[1]
            chi = (S[1, 1] * n0 * n0 - (S[0, 1] + S[1, 0]) * n0 * n1 + S[0, 0] * n1 * n1) / det
            assert abs(chi / CHI2 - 1) > 1e-12, f"candidate ({j}, {i}) on the chi-square gate"
            ok = chi < CHI2 and HP < j < nCols - HP and HP < i < nRows - HP
            out.append((j, i, ok))
    return out, hsx, hsy


def zncc_exact(patch, windows):
    """exact centred sums of a (169,) integer patch against (m, 169) integer windows -> (num, va, vb) as Python ints"""
    a = patch.astype(np.int64)
    B = windows.astype(np.int64)
    sa, saa = int(a.sum()), int((a * a).sum())
    sb, sbb, sab = B.sum(1), (B * B).sum(1), B @ a
    va = 169 * saa - sa * sa
    return [(169 * int(sab[k]) - sa * int(sb[k]), va, 169 * int(sbb[k]) - int(sb[k]) ** 2) for k in range(B.shape[0])]


def search_reference(img, h, S, patch, cam=CAM9):
    """The exact active search of one feature.  Returns dict(kind, allowed): kind 'none' (no match), 'one' (allowed = [(j, i)]) or
    'band' (allowed = the candidates within 1e-12 of the best score, any of which may be returned)."""
    nRows, nCols = int(cam[2]), int(cam[3])
    if not lmax_of(S) < MAX_EIG:
        return dict(kind="none", why="eig")
    assert abs(lmax_of(S) / MAX_EIG - 1) > 1e-12
    if not (HP < h[0] < nCols - HP and HP < h[1] < nRows - HP):  # zero predicted patch (src/Tracking.cpp:174-175, 275): NaN scores
        return dict(kind="none", why="border")
    cands, _, _ = gate(h, S, cam)
    acc = [(j, i) for j, i, ok in cands if ok]
    if not acc:
        return dict(kind="none", why="no candidate")
    W = np.stack([img[i - HP:i + HP + 1, j - HP:j + HP + 1].reshape(-1) for j, i in acc])
    sums = zncc_exact(np.asarray(patch).reshape(-1), W)
    if sums[0][1] == 0 or sums[0][2] == 0:  # NaN in slot 0 is sticky (Eigen's maxCoeff, Q10)
        return dict(kind="none", why="slot0")
    keys = [None if va == 0 or vb == 0 else Fraction(num * abs(num), va * vb) for num, va, vb in sums]
    best = max(k for k in keys if k is not None)
    num, va, vb = sums[keys.index(best)]
    corr = num / math.sqrt(va * vb)
    assert abs(corr / CORR_THR - 1) > 1e-12, "best score on the correlation threshold"
    if not (num > 0 and 25 * num * num > 16 * va * vb):
        return dict(kind="none", why="threshold")
    near = [c for c, k, (n_, a_, b_) in zip(acc, keys, sums) if k is not None and n_ / math.sqrt(a_ * b_) >= corr * (1 - 1e-12)]
    if len(near) == 1:
        return dict(kind="one", allowed=near)
    wins = {tuple(img[i - HP:i + HP + 1, j - HP:j + HP + 1].reshape(-1)) for j, i in near}
    if len(wins) == 1:  # identical windows: bitwise identical scores, the first visited wins
        return dict(kind="one", allowed=near[:1], tied=len(near), pair=near)
    return dict(kind="band", allowed=near)


@pytest.mark.parametrize("seed", range(6))
def test_exact_zncc_matches_corrcoef(seed):
    """The exact centred sums give the scores of oracle_py.corrcoef (Converter::corrcoef_opencv) to 1e-12 on random windows, including
    constant and near-constant ones."""
    from oracle import oracle_py as O

    rng = np.random.default_rng([seed, 25])
    m = 40
    M = rng.integers(0, 256, (169, m + 1)).astype(np.float64)
    M[:, 3] = 17.0
    M[:, 5] = M[:, 0] + 30
    M[:5, 7] = 255.0
    ref = O.corrcoef(M, row0_only=True)[0, 1:]
    sums = zncc_exact(M[:, 0], M[:, 1:].T)
    for k, (num, va, vb) in enumerate(sums):
        if vb == 0:
            assert np.isnan(ref[k])
            continue
        assert abs(num / math.sqrt(va * vb) - ref[k]) <= 1e-12, k


# The search scenes.  Features sit on a grid whose search regions (<= 2 * 20 + 1 candidates + a 13-pixel window) do not overlap, so
# what is planted for one feature cannot change another's answer.  Each feature is (name, h, S, patch) and the scene also edits the
# image.  Patches and images are integers.
GRID_X = [33, 88, 143, 198, 253]  # + jitter < 1: regions of half-width 26.5 stay apart and inside the image
GRID_Y = [33, 88, 143, 198]


def sdiag(hsx, hsy, c=0.0):
    """S with window half-widths (hsx, hsy) (2 sqrt(S_ii) = hs - 0.5, or just under the eigenvalue gate for 20) and correlation c"""
    sx = (hsx - 0.5) ** 2 / 4 if hsx < 20 else 99.99
    sy = (hsy - 0.5) ** 2 / 4 if hsy < 20 else 99.99
    o = c * math.sqrt(sx * sy)
    S = np.array([[sx, o], [o, sy]])
    if c and not lmax_of(S) < 99.0:
        S[0, 1] = S[1, 0] = 0.0
    return S


def S_with_lmax(L, a=99.9, d=1.3):
    b = math.sqrt((L - (a + d) / 2) ** 2 - ((a - d) / 2) ** 2)
    return np.array([[a, b], [b, d]])


class Scene:
    def __init__(self, seed, rows=ROWS, cols=COLS):
        self.rng = np.random.default_rng([seed, 26])
        self.img = self.rng.integers(0, 256, (rows, cols)).astype(np.uint8)
        self.feats = []  # (name, h, S, patch or ("copy", j, i, noise))
        self.slots = [(x, y) for y in GRID_Y for x in GRID_X]

    def h_at(self, slot):
        x, y = self.slots[slot]
        return np.array([x + self.rng.choice([0.3, -0.2, 0.15, -0.35]), y + self.rng.choice([0.25, -0.3, 0.1, -0.15])])

    def accepted(self, h, S):
        return [(j, i) for j, i, ok in gate(h, S)[0] if ok]

    def block(self, lo=0, hi=256):
        return self.rng.integers(lo, hi, (13, 13))

    def put(self, j, i, blk):
        self.img[i - HP:i + HP + 1, j - HP:j + HP + 1] = blk

    def add_copy(self, name, h, S, target=None, noise=0):
        acc = self.accepted(h, S)
        t = acc[self.rng.integers(len(acc))] if target is None else target
        assert t in acc
        self.feats.append((name, h, S, ("copy", t[0], t[1], noise)))
        return t

    def finish(self):
        """resolve copied patches (after every image edit) -> (image, [(name, h, S, patch float64 13 x 13)])"""
        out = []
        for name, h, S, p in self.feats:
            if isinstance(p, tuple):
                _, j, i, noise = p
                w = self.img[i - HP:i + HP + 1, j - HP:j + HP + 1].astype(np.int64)
                if noise:
                    w = np.clip(w + self.rng.integers(-noise, noise + 1, w.shape), 0, 255)
                p = w
            out.append((name, h, S, np.asarray(p, np.float64)))
        self.img.flags.writeable = False
        return self.img, out


def shape_scenes():
    """Every hsx and every hsy in 1..20 (each value paired once with itself and once with 21 - itself): both residues of the strip
    padding (ncy = 2 hsy + 1 is 1 or 3 mod 4), 41 x 41 candidates at S just under max_ellipse_eig; perfect copies and copies with +-3 of noise."""
    pairs = [(k, k) for k in range(1, 21)] + [(k, 21 - k) for k in range(1, 21)]
    scenes = []
    for s in range(2):
        sc = Scene(100 + s)
        for slot, (hx, hy) in enumerate(pairs[20 * s:20 * s + 20]):
            h = sc.h_at(slot)
            S = sdiag(hx, hy, c=0.3 if slot % 3 == 1 else 0.0)
            sc.add_copy(f"hs{hx}x{hy}", h, S, noise=3 if slot % 2 else 0)
        scenes.append(sc.finish())
    return scenes


def rule_scene(seed=200):
    """Ties, NaN rules, gates and borders, one per grid slot (and eight on the image border)."""
    sc = Scene(seed)
    S15 = sdiag(15, 15)
    slot = iter(range(20))

    def plant_pair(name, d1, d2, offset=0):
        h = sc.h_at(next(slot))
        cx, cy = c_round(h[0]), c_round(h[1])
        blk = sc.block(0, 256 - offset)
        p1, p2 = (cx + d1[0], cy + d1[1]), (cx + d2[0], cy + d2[1])
        acc = sc.accepted(h, S15)
        assert p1 in acc and p2 in acc
        sc.put(*p1, blk)
        sc.put(*p2, blk + offset)
        sc.feats.append((name, h, S15, blk))

    plant_pair("identical-same-x", (0, -7), (0, 7))  # the smaller y is visited first
    plant_pair("identical-diff-x", (7, -7), (-7, 7))  # the smaller x is visited first, although its y is larger
    plant_pair("identical-same-warp", (7, 0), (-7, 0))  # two lanes of one warp: the shuffle's tie rule decides
    plant_pair("exact-tie-b+c", (-7, 0), (7, 0), offset=40)  # tied in exact arithmetic, decided by rounding: either may win
    plant_pair("exact-tie-b+c-y", (0, 7), (0, -7), offset=9)
    # a constant window at the first accepted candidate: NaN in slot 0 is sticky -> no match, although a perfect copy exists
    h = sc.h_at(next(slot))
    acc = sc.accepted(h, S15)
    sc.put(*acc[0], np.full((13, 13), 77))
    sc.add_copy("const-slot0", h, S15, target=acc[-1])
    # a constant window later in the order must not block the match
    h = sc.h_at(next(slot))
    acc = sc.accepted(h, S15)
    sc.put(*acc[len(acc) // 3], np.full((13, 13), 255))
    sc.add_copy("const-later", h, S15, target=acc[-3])
    # a constant predicted patch: every score is NaN
    h = sc.h_at(next(slot))
    sc.feats.append(("const-patch", h, S15, np.full((13, 13), 128)))
    # no candidate passes the chi-square gate (S tiny, h off the pixel grid): no match, nothing written
    h = sc.h_at(next(slot))
    sc.feats.append(("no-candidate", h, np.array([[0.001, 0.0], [0.0, 0.0012]]), sc.block()))
    # the eigenvalue gate, 1e-9 below and above 100 (hsx = 20, off-diagonal S)
    for nm, L in (("eig-below", 100 * (1 - 1e-9)), ("eig-above", 100 * (1 + 1e-9))):
        h = sc.h_at(next(slot))
        sc.add_copy(nm, h, S_with_lmax(L))
    # the best candidate below corr_threshold (a copy drowned in noise): no match
    h = sc.h_at(next(slot))
    sc.add_copy("below-threshold", h, sdiag(4, 4), noise=255)
    # h within half a patch of the border: the kernel returns at once (the reference's predicted patch is zero there)
    for nm, hb in (("border-left", (5.8, 120.3)), ("border-right", (COLS - 5.7, 100.3)), ("border-top", (120.3, 5.9)),
                   ("border-bottom", (100.3, ROWS - 5.8))):
        sc.feats.append((nm, np.array(hb), sdiag(3, 3), sc.block()))
    # candidates cut by the border rule j > 6, j < nCols - 6, i > 6, i < nRows - 6 (the window staging reads outside the image there)
    for nm, hb, t in (("cut-left", (8.3, 60.3), (7, 61)), ("cut-right", (COLS - 8.3, 60.3), (COLS - 7, 59)),
                      ("cut-top", (60.3, 8.3), (61, 7)), ("cut-bottom", (60.3, ROWS - 8.3), (59, ROWS - 7))):
        sc.add_copy(nm, np.array(hb), sdiag(10, 10), target=t)
    return sc.finish()


def search_thread(h, S, j, i):
    """(warp, lane, strip) of the k_search thread that scores candidate (j, i): strips of kStrip = 4 rows, strip = jx + ncx (iy / 4),
    64 threads striding over the strips"""
    _, hsx, hsy = gate(h, S)
    jx, iy = j - (c_round(h[0]) - hsx), i - (c_round(h[1]) - hsy)
    strip = jx + (2 * hsx + 1) * (iy // 4)
    return (strip % 64) // 32, strip % 32, strip


EXPECT_KIND = {"identical-same-warp": "one", "identical-same-x": "one", "identical-diff-x": "one", "exact-tie-b+c": "band", "exact-tie-b+c-y": "band", "const-slot0": "none",
               "const-later": "one", "const-patch": "none", "no-candidate": "none", "eig-below": "one", "eig-above": "none",
               "below-threshold": "none", "border-left": "none", "border-right": "none", "border-top": "none", "border-bottom": "none",
               "cut-left": "one", "cut-right": "one", "cut-top": "one", "cut-bottom": "one"}


@functools.lru_cache(maxsize=None)
def search_scenes():
    """{name: (image, feats, refs)}: two shape scenes and the rule scene with the exact reference of every feature"""
    out = {}
    named = [(f"shapes{k}", sc) for k, sc in enumerate(shape_scenes())] + [("rules", rule_scene())]
    for name, (img, feats) in named:
        out[name] = (img, feats, [search_reference(img, h, S, p) for _, h, S, p in feats])
    return out


def test_search_scenes_reach_their_edges():
    """Every shape case is decided and matched at its copy; every rule case has the outcome it was built for; all margins hold."""
    sc = search_scenes()
    seen_x, seen_y = set(), set()
    for name in ("shapes0", "shapes1"):
        img, feats, refs = sc[name]
        for (nm, h, S, p), r in zip(feats, refs):
            assert r["kind"] == "one", (nm, r)
            _, hsx, hsy = gate(h, S)
            seen_x.add(hsx)
            seen_y.add(hsy)
    assert seen_x == seen_y == set(range(1, 21))
    assert {(2 * hy + 1) % 4 for hy in seen_y} == {1, 3}  # ncy is odd: strips padded by 3 and by 1 rows
    img, feats, refs = sc["rules"]
    for (nm, h, S, p), r in zip(feats, refs):
        assert r["kind"] == EXPECT_KIND[nm], (nm, r)
    r = dict(zip([f[0] for f in feats], refs))
    assert r["identical-same-x"]["tied"] == 2 and r["identical-diff-x"]["tied"] == 2 and r["identical-same-warp"]["tied"] == 2
    # the pairs reach both levels of the arg-max: lanes of one warp (shuffle) and two warps (the block's shared-memory step)
    fs = {nm: (h, S) for nm, h, S, _ in feats}
    for nm, same_warp in (("identical-same-warp", True), ("identical-same-x", False), ("identical-diff-x", False)):
        h, S = fs[nm]
        (w1, l1, _), (w2, l2, _) = (search_thread(h, S, *c) for c in r[nm]["pair"])
        assert (w1 == w2) == same_warp and l1 != l2, nm
    assert len(r["exact-tie-b+c"]["allowed"]) == 2 and len(r["exact-tie-b+c-y"]["allowed"]) == 2
    assert r["const-slot0"]["why"] == "slot0" and r["no-candidate"]["why"] == "no candidate" and r["eig-above"]["why"] == "eig"
    assert r["below-threshold"]["why"] == "threshold"
    cut = [gate(h, S)[0] for nm, h, S, p in feats if nm.startswith("cut")]
    assert all(any(not ok and (j <= HP or j >= COLS - HP or i <= HP or i >= ROWS - HP) for j, i, ok in c) for c in cut)


# ---- snapshot patching: inject h, S, has_h and the predicted patch ----------------------------------------------------------------
def patch_snapshot(buf, k, **arrays):
    """a copy of snapshot `buf` with record arrays of its filter k replaced (names of capi._CK_RECORDS), at the offsets
    capi.read_checkpoint walks"""
    out = np.array(buf, dtype=np.uint8, copy=True)
    e = 160 + 32 * k
    boff = int(out[e:e + 8].view("<u8")[0])
    n, N = (int(v) for v in out[e + 16:e + 24].view("<i4"))
    o = boff + 16
    for name, dt, shape, unit in capi._CK_RECORDS:
        cnt = (n if unit == "n" else N) * int(np.prod(shape, dtype=np.int64))
        nbytes = cnt * np.dtype(dt).itemsize
        if name in arrays:
            v = np.ascontiguousarray(arrays.pop(name), dtype=dt).reshape(-1)
            assert v.size == cnt, (name, v.size, cnt)
            out[o:o + nbytes] = v.view(np.uint8)
        o += (nbytes + 15) & ~15
    assert not arrays, f"unknown record arrays {list(arrays)}"
    return out


def test_snapshot_patch_changes_exactly_the_intended_bytes():
    """Patching S, h, has_h and the patches of one filter of the golden snapshot changes only bytes inside those arrays, and
    read_checkpoint returns the patched arrays and every other array unchanged."""
    import os

    buf = np.fromfile(os.path.join(os.path.dirname(__file__), "golden", "checkpoint_v1.bin"), dtype=np.uint8)
    _, before = capi.read_checkpoint(buf)
    k = len(before) - 1
    N = before[k]["N"]
    rng = np.random.default_rng(27)
    new = dict(S=rng.standard_normal((N, 2, 2)), h=rng.standard_normal((N, 2)), has_h=np.arange(N) % 2 == 0,
               patches=rng.integers(0, 256, (N, 13, 13)).astype(np.float32))
    out = patch_snapshot(buf, k, **{a: b.copy() for a, b in new.items()})
    _, after = capi.read_checkpoint(out)
    for j, (fb, fa) in enumerate(zip(before, after)):
        for name in fb:
            if j == k and name in new:
                assert np.array_equal(fa[name], new[name]), name
            else:
                assert np.array_equal(fa[name], fb[name]), (j, name)
    changed = np.flatnonzero(out != buf)
    total = sum(np.asarray(v).nbytes if v.dtype != bool else N for v in new.values())
    assert 0 < changed.size <= total


def search_handle(members, Nmax=None, cam=CAM9):
    """A handle whose filter b holds members[b] = feats list [(name, h, S, patch)] (with optional has_h mask as members[b][1]):
    uploads a placeholder map of the right size, then injects h, S, has_h and the patches through a snapshot.  z is set to -7 and
    ic to 0 so that a write by the search shows."""
    B = len(members)
    Nmax = Nmax or max(len(m[0]) for m in members)
    f = capi.Filter(cam, Nmax, batch=B)
    for b, (feats, _) in enumerate(members):
        N = len(feats)
        n = 13 + 6 * N
        x = np.zeros(n)
        x[3] = 1.0
        f.upload_state(x, np.eye(n), feat_types=np.zeros(N, np.int32), b=b)
    buf = f.save()
    for b, (feats, has_h) in enumerate(members):
        N = len(feats)
        buf = patch_snapshot(buf, b, h=np.array([h for _, h, _, _ in feats]), S=np.array([S for _, _, S, _ in feats]),
                             has_h=has_h if has_h is not None else np.ones(N, bool), patches=np.array([p for *_, p in feats]),
                             z=np.full((N, 2), -7.0), ic=np.zeros(N, bool))
    f.load(buf)
    return f


def check_search(f, b, feats, refs, has_h=None, what=""):
    fg = f.features(b)
    for k, ((nm, h, S, p), r) in enumerate(zip(feats, refs)):
        ic, z = bool(fg["ic"][k]), tuple(fg["z"][k])
        tag = f"{what} feature {k} ({nm})"
        if (has_h is not None and not has_h[k]) or r["kind"] == "none":
            assert not ic and z == (-7.0, -7.0), f"{tag}: expected no match, got {z}"
        else:
            assert ic, f"{tag}: expected a match in {r['allowed']}"
            assert z in [(float(j), float(i)) for j, i in r["allowed"]], f"{tag}: {z} not in {r['allowed']}"


@pytest.mark.gpu
@pytest.mark.parametrize("scene", ["shapes0", "shapes1", "rules"])
def test_search_scene(scene):
    """One filter per scene, its image bound alone (share = 0)."""
    img, feats, refs = search_scenes()[scene]
    f = search_handle([(feats, None)])
    try:
        f.set_image(img)
        f.match()
        check_search(f, 0, feats, refs, what=scene)
    finally:
        f.close()


def padded(img, stride, fill=255):
    out = np.full((img.shape[0], stride), fill, np.uint8)
    out[:, :img.shape[1]] = img
    return out


@pytest.mark.gpu
def test_search_batch_own_images_with_stride_and_heterogeneous_N():
    """Three filters with their own images (share = 0), the rule scene's read through a stride of 352 with bright padding, and
    heterogeneous N: filter 2 holds the first 13 shape features with every third one's has_h cleared (left untouched)."""
    sc = search_scenes()
    img0, f0, r0 = sc["shapes0"]
    img1, f1, r1 = sc["rules"]
    f2, r2 = f0[:13], r0[:13]
    hh = np.arange(13) % 3 != 0
    f = search_handle([(f0, None), (f1, None), (f2, hh)])
    try:
        f.set_image(img0, b=0)
        f.set_image(padded(img1, 352), b=1, cols=COLS)
        f.set_image(img0, b=2)
        f.match()
        check_search(f, 0, f0, r0, what="filter 0")
        check_search(f, 1, f1, r1, what="filter 1")
        check_search(f, 2, f2, r2, has_h=hh, what="filter 2")
    finally:
        f.close()


@pytest.mark.gpu
def test_search_batch_shared_image():
    """One image shared by a batch of three (share = 1): the rule scene whole, its first 7 features, and its last 9."""
    img, feats, refs = search_scenes()["rules"]
    parts = [(feats, refs), (feats[:7], refs[:7]), (feats[-9:], refs[-9:])]
    f = search_handle([(p, None) for p, _ in parts])
    try:
        f.set_image(img, b=1, share=True)
        f.match()
        for b, (p, r) in enumerate(parts):
            check_search(f, b, p, r, what=f"filter {b}")
    finally:
        f.close()


@pytest.mark.gpu
def test_search_on_predicted_S_against_the_oracle():
    """S from a real k_predict (whose off-diagonals need not be bitwise equal): the device's matches equal the exact reference on the
    device's h and S, and the C++ oracle's Tracking::matching on the same state, image and patches."""
    from oracle import oracle_py as O

    cam, types, x, P = visible_map(40, seed=7, cart_every=0)
    N = len(types)
    rng = np.random.default_rng(28)
    img = rng.integers(0, 256, (ROWS, COLS)).astype(np.uint8)
    f = capi.Filter(cam, N)
    try:
        f.upload_state(x, P, feat_types=types, prior=True)
        f.predict_measurements()
        fg = f.features()
        patches = np.zeros((N, 13, 13))
        feats = []
        for k in range(N):
            h, S = fg["h"][k], fg["S"][k]
            p = np.zeros((13, 13))
            if fg["has_h"][k] and lmax_of(S) < MAX_EIG and HP < h[0] < COLS - HP and HP < h[1] < ROWS - HP:
                acc = [(j, i) for j, i, ok in gate(h, S)[0] if ok]
                if acc:
                    j, i = acc[rng.integers(len(acc))]
                    p = img[i - HP:i + HP + 1, j - HP:j + HP + 1].astype(np.float64)
            patches[k] = p
            feats.append((f"f{k}", h, S, p))
        refs = [search_reference(img, h, S, p) if fg["has_h"][k] else dict(kind="none") for k, (_, h, S, p) in enumerate(feats)]
        assert sum(r["kind"] == "one" for r in refs) > N // 2 and not any(r["kind"] == "band" for r in refs)
        f.upload_patches(patches)
        f.set_image(img)
        f.match()
        check_search(f, 0, feats, refs, has_h=fg["has_h"])
        o = O.OracleFilter(cam, fast_corr=True)
        for k in range(N):
            o.add_feature(int(types[k]), None, patches[k], np.zeros(3), np.eye(3), np.zeros(2))
        o.set_state(x, P, prior=True)
        o.search_ic_matches(img)
        fo, fd = o.features(), f.features()
        assert np.array_equal(fo["ic"], fd["ic"])
        assert np.array_equal(fo["z"][fo["ic"]], fd["z"][fd["ic"]])
    finally:
        f.close()


# ---- image binding: binding one filter's image never changes what another filter reads -----------------------------------------
def two_scene_handle():
    sc = search_scenes()
    a, b = sc["shapes0"], sc["shapes1"]
    return a, b, search_handle([(a[1], None), (b[1], None)])


@pytest.mark.gpu
def test_set_image_strides_of_different_calls_do_not_overlap():
    """Filter 0 bound with stride 384, then filter 1 with stride 320: filter 1's copy must not land inside filter 0's image."""
    a, b, f = two_scene_handle()
    try:
        f.set_image(padded(a[0], 384), b=0, cols=COLS)
        f.set_image(b[0], b=1)
        f.match()
        check_search(f, 0, a[1], a[2], what="filter 0")
        check_search(f, 1, b[1], b[2], what="filter 1")
    finally:
        f.close()


@pytest.mark.gpu
def test_set_image_growth_keeps_the_other_filters_images():
    """Filter 0 bound with stride 320, then filter 1 with stride 448 (more than the batch's staging held): filter 0 keeps reading its
    own image."""
    a, b, f = two_scene_handle()
    try:
        f.set_image(a[0], b=0)
        f.set_image(padded(b[0], 448), b=1, cols=COLS)
        f.match()
        check_search(f, 0, a[1], a[2], what="filter 0")
        check_search(f, 1, b[1], b[2], what="filter 1")
    finally:
        f.close()


@pytest.mark.gpu
def test_set_image_own_after_shared():
    """A shared binding (image b for both), then filter 0 bound to its own image a: filter 1 still reads the shared image b."""
    a, b, f = two_scene_handle()
    try:
        f.set_image(b[0], b=0, share=True)
        f.set_image(a[0], b=0)
        f.match()
        check_search(f, 0, a[1], a[2], what="filter 0")
        check_search(f, 1, b[1], b[2], what="filter 1 (shared image)")
    finally:
        f.close()


# ---- the eigenvalue gate bounds the search window ----------------------------------------------------------------------------------
def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def lmax_variants(a, b, d):
    """k_search's lmax = 0.5 (a + d) + sqrt(0.25 (a - d)(a - d) + b b) under every contraction of its products into FMAs"""
    t = 0.25 * (a - d)
    inner = [t * (a - d) + b * b, _fma(t, a - d, b * b), _fma(b, b, t * (a - d))]
    out = []
    for v in inner:
        s = math.sqrt(v)
        out += [0.5 * (a + d) + s, _fma(0.5, a + d, s)]
    return out


def test_eigenvalue_gate_bounds_the_search_window():
    """Wherever k_search accepts S (lmax < 100, however its expression is contracted), ceil(2 sqrt(S_ii)) <= 20 = kMaxHalfSearch as
    the kernel computes it, so no accepted feature can be dropped for want of window space.  The sample crowds the boundary: diagonals
    within a few ulps of 100 and of 90.25 (where the half-width steps from 19 to 20), off-diagonals from 0 to large."""
    rng = np.random.default_rng(29)
    vals = []
    for base in (100.0, 90.25, 99.99999999999):
        v = base
        for _ in range(6):
            vals.append(v)
            v = float(np.nextafter(v, 200.0))
        v = base
        for _ in range(6):
            v = float(np.nextafter(v, 0.0))
            vals.append(v)
    vals += list(rng.uniform(95, 100.5, 200)) + list(rng.uniform(-5, 5, 20))
    offs = [0.0, 5e-324, 1e-300, 1e-160, 1e-12, 1e-8, 1e-4, 0.1, 3.0]
    accepted = 0
    for a in vals:
        for d in vals[::7]:
            for b in offs + list(rng.uniform(0, 20, 3)):
                if any(lm < MAX_EIG for lm in lmax_variants(a, b, d)):
                    accepted += 1
                    for s in (a, d):
                        if s >= 0:
                            assert math.ceil(2 * math.sqrt(s)) <= 20, (a, b, d)
    assert accepted > 1000


def test_create_refuses_max_ellipse_eig_outside_0_100():
    """max_ellipse_eig must be finite and in (0, 100]: the search window is sized for lmax < 100.  Refused before any device work."""
    for bad in (100.0000001, 1e3, math.inf, math.nan, 0.0, -1.0):
        with pytest.raises(capi.RslamError, match="max_ellipse_eig"):
            capi.Filter(CAM9, 4, max_ellipse_eig=bad)
