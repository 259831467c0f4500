"""The 1-point RANSAC kernels -- k_ransac_compact / k_ransac_compact_hyp, k_ransac_hyp, k_ransac_support, k_ransac_select and the sweep
kernels k_sweep_compact, k_sweep_prep and k_sweep_reduce -- against float64 and exact references, at the edges where they branch.

In a whole frame the data decide the number of matches, their order and the draws.  Here the state is uploaded (rslam_upload_state),
rslam_predict_measurements produces h, S, Hc and Hf (k_predict, verified against float64 in test_gpu_track_kernels.py), the matches z
and ic are chosen by the test (rslam_set_matches) and so are the uniform draws.  Each case names the edge it exists for.

References:
- support: src/Tracking.cpp:419-477 in float64 from the 13 structurally non-zero columns of H_p, for any mix of feature types (the
  feature offsets need not be 13 + 6 j).  A decision may differ from the kernel's only where the float64 residual lies within 1e-9 px
  of std_z (the project's band rule); planted decisions are exact.
- selection: select_reference, a restatement of the reference's adaptive loop (oracle/rslam_oracle.cpp:712-790, src/Tracking.cpp:403-537)
  with its logarithms taken by math.log, which is libm's log as std::log is in the reference; checked against the C++ oracle below.
  Status, hyp_run, best_support, n_hyp and the winner are exact, and li is exactly the winner's mask.

The library's convention for a draw u = 1.0 (the reference's quirk Q8 indexes one past the last match there): it lands on the last match,
floor(u nIC) clamped to nIC - 1, on the resolved and on the direct path of k_ransac_select alike."""
import functools
import hashlib
import math

import numpy as np
import pytest

from oracle import np_oracle as NP
from ransac_slam_b200 import capi, synth
from tests.test_gpu_track_kernels import layout, undistort

CAM9 = synth.Camera().as9()
Q_ALL, Q1 = 0x7, 0x1
ROWS, COLS = 240, 320


def quirks(q1):
    return Q_ALL if q1 else Q_ALL & ~Q1


# ---- references ----------------------------------------------------------------------------------------------------------------------
def support_reference(x, P, offs, Hc, Hf, h, z, p, ids, q1, inv=True, cam=CAM9):
    """Hypothesis from feature p (inverse depth), scored on the matched features ids (inverse depth, in match order).  Returns
    (residuals, hd (m, 2), hc (3, m), x_i).  inv: K from the explicit inverse of S, else from a solve."""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = cam
    o = int(offs[p])
    Hs = np.concatenate([Hc[p], Hf[p]], axis=1)  # 2 x 13
    Pc = np.concatenate([P[:, 0:7], P[:, o:o + 6]], axis=1)
    sel = list(range(7)) + list(range(o, o + 6))
    S = Hs @ Pc[sel, :] @ Hs.T + np.eye(2)
    nu = z[p] - h[p]
    xi = x + (Pc @ (Hs.T @ (np.linalg.inv(S) @ nu)) if inv else Pc @ (Hs.T @ np.linalg.solve(S, nu)))
    mo = offs[ids]
    m = len(ids)
    ri = np.stack([xi[mo], xi[mo + 1], xi[mo + 2]], axis=0)
    if q1:  # quirk Q1: the angles of match c are entries (2c, 2c+1) of the stacked positions of all matches
        riv = ri.T.reshape(-1)
        a0, a1 = riv[0:2 * m:2], riv[1:2 * m:2]
    else:
        a0, a1 = xi[mo + 3], xi[mo + 4]
    rho = xi[mo + 5]
    mi = np.stack([np.cos(a1) * np.sin(a0), -np.sin(a1), np.cos(a1) * np.cos(a0)], axis=0)
    v = (ri - xi[0:3, None]) * rho[None, :] + mi
    hc = NP.q2r(xi[3:7]).T @ v
    himg = np.stack([f / dx * hc[0] / hc[2] + Cx, f / dx * hc[1] / hc[2] + Cy], axis=1)
    hd = NP.distort_fm(cam, himg)
    return np.sqrt(((z[ids] - hd) ** 2).sum(axis=1)), hd, hc, xi


def n_hyp_of(s, nic, p):
    """(int) ceil(log(1 - p) / log(1 - (1 - epsilon))) with epsilon = 1 - s / nIC, libm's log, log(0) = -inf"""
    eps = 1 - s / nic
    d = 1 - (1 - eps)
    return int(math.ceil(math.log(1 - p) / (math.log(d) if d > 0 else -math.inf)))


def draw_t(u, nic):
    return min(int(math.floor(u * nic)), nic - 1)


def select_reference(sup, nic, u01, p=0.99, n_hyp0=1000):
    """The reference's loop (oracle/rslam_oracle.cpp:712-790) over the supports sup[t] of the distinct hypotheses."""
    if nic == 0:  # Q9
        return dict(status=1, hyp_run=0, best_support=0, n_hyp=n_hyp0, winner=-1)
    n_hyp, best, win, run, status = n_hyp0, 0, -1, 0, 0
    i = 0
    while i < n_hyp:
        if i >= len(u01):
            status = 3
            break
        s = int(sup[draw_t(u01[i], nic)])
        run = i + 1
        if s > best:
            best, win = s, i
            n_hyp = n_hyp_of(s, nic, p)
            if n_hyp == 0:
                break
        if i > n_hyp:
            break
        i += 1
    return dict(status=status, hyp_run=run, best_support=best, n_hyp=n_hyp, winner=win)


def band_check(got, res, std_z, what):
    diff = got != (res < std_z)
    assert (np.abs(res[diff] - std_z) <= 1e-9).all(), f"{what}: {int(diff.sum())} decisions differ outside the 1e-9 px band"


# ---- the restatement against the C++ oracle (CPU) ------------------------------------------------------------------------------------
def oracle_case(kind):
    from oracle import oracle_py as O
    from tests import helpers as H

    if kind == "q1":
        cam, x, P, z, ic = H.q1_consistent_state(40, seed=5)
        o = O.OracleFilter(cam.as9())
        for _ in range(40):
            o.add_feature(0, None, np.zeros((13, 13)), np.zeros(3), np.eye(3), np.zeros(2))
        o.set_state(x, P, prior=True)
        o.search_ic_matches(None)
        o.set_matches(z, ic)
        return o, cam.as9(), x, P, True, np.random.default_rng(7).random(3000)
    N, seed = (30, 54) if kind == "spd30" else (40, 91)
    scene, x, P = synth.random_spd_state(N, seed=seed)
    seq = synth.make_sequence(scene, T=1, seed=seed + 5, t0=3)
    o = H.oracle_from(scene, x, P, quirks=O.Q_ALL & ~O.Q1)
    o.search_ic_matches(seq.images[0])
    return o, scene.cam.as9(), x, P, False, seq.u01[0]


@pytest.mark.parametrize("kind", ["spd30", "spd40", "q1"])
def test_select_reference_matches_the_cpp_oracle(kind):
    """select_reference over np_oracle.hypothesis_support's supports reproduces the C++ oracle's status, counters and li flags."""
    o, cam, x, P, q1, u = oracle_case(kind)
    f = o.features()
    ic = np.flatnonzero(f["ic"])
    types = np.zeros(len(f["ic"]), int)
    sup, masks = [], []
    for p in ic:
        s, inl, res = NP.hypothesis_support(cam, x, P, types, o.H_dense(p), f["h"][p], f["z"][p], f["z"], f["ic"], q1=q1)
        assert (np.abs(res - 1.0) > 1e-9).all()
        sup.append(s)
        masks.append(inl)
    exp = select_reference(sup, ic.size, u)
    rc, info = o.ransac_hypotheses(u)
    assert (rc, info["hyp_run"], info["best_support"], info["n_hyp"]) == (exp["status"], exp["hyp_run"], exp["best_support"], exp["n_hyp"])
    assert exp["best_support"] > 0
    li = o.features()["li"]
    assert (li[ic] == masks[draw_t(u[exp["winner"]], ic.size)]).all()


# ---- n_hyp rounding (CPU scan) -----------------------------------------------------------------------------------------------------
def near_integer_pairs(p, nic_max=8192, ulps=4):
    """(s, nIC), 1 <= s < nIC <= nic_max, whose ratio log(1 - p) / log(1 - (1 - epsilon)) (libm) lies within `ulps` ulps of an integer.
    numpy screens at 64 ulps; math.log decides."""
    out = []
    la = math.log(1 - p)
    for nic in range(2, nic_max + 1):
        s = np.arange(1, nic)
        d = 1 - (1 - (1 - s / nic))
        r = la / np.log(d)
        for sv in s[np.abs(r - np.rint(r)) <= 64 * np.spacing(r)]:
            eps = 1 - int(sv) / nic
            rv = la / math.log(1 - (1 - eps))
            if abs(rv - round(rv)) <= ulps * math.ulp(rv):
                out.append((int(sv), nic))
    return out


# p -> (pair count, sha1 of the list's repr, {reduced fraction: ratio})
NHYP_PINS = {0.9: (819, "aecddeda72abecbd", {(9, 10): 1.0}),
             0.99: (900, "053edbfe0a1f1256", {(9, 10): 1.9999999999999996, (99, 100): 1.0}),
             0.999: (827, "3d19ae97980e7b51", {(9, 10): 2.999999999999999, (999, 1000): 1.0})}


@pytest.mark.parametrize("p", sorted(NHYP_PINS))
def test_n_hyp_near_integer_scan(p):
    """The pairs where n_hyp = ceil(ratio) hangs on the last bits of two logarithms: two families per p (s / nIC = 9 / 10, and
    (1 - (1 - p)) exactly, where both logs see the same argument and the ratio is exactly 1).  Pinned; the GPU test checks members."""
    pairs = near_integer_pairs(p)
    cnt, digest, fams = NHYP_PINS[p]
    assert len(pairs) == cnt and hashlib.sha1(repr(pairs).encode()).hexdigest()[:16] == digest
    seen = {}
    for s, nic in pairs:
        g = math.gcd(s, nic)
        seen[(s // g, nic // g)] = math.log(1 - p) / math.log(1 - (1 - (1 - s / nic)))
    assert seen == fams


# ---- scenes --------------------------------------------------------------------------------------------------------------------------
def q1_angles(anchors, matched, th, ph):
    """write the matches' angles into entries (2c, 2c+1) of their stacked positions, so that quirk Q1 reads the true angles"""
    m = len(matched)
    st = anchors[matched].reshape(-1).copy()
    st[0:2 * m:2] = th[matched]
    st[1:2 * m:2] = ph[matched]
    anchors[matched] = st.reshape(m, 3)


@functools.lru_cache(maxsize=2)
def geom_scene(N, m, n_cart, seed=0, outliers=0.25, gross=0.0, cam_sd=1.0):
    """N features, n_cart of them cartesian and unmatched, m inverse-depth ones matched, interleaved with unmatched ones.  The matches'
    stacked positions carry their angles (consistent under Q1 on and off).  z = h + N(0, 0.4 px), a fraction moved by 3..15 px and a
    fraction by 40..80 px; the first and the last match are kept clean.  Returns dict(types, x, P, z, ic, matched, offs), read only."""
    rng = np.random.default_rng([N, m, n_cart, seed, 41])
    types = np.zeros(N, np.int32)
    if n_cart:
        types[np.linspace(1, N - 1, n_cart).astype(int)] = 1
    idp = np.flatnonzero(types == 0)
    assert idp.size >= m
    matched = np.sort(rng.choice(idp, m, replace=False))
    offs, sizes, n = layout(types)
    x = np.zeros(n)
    x[0:3] = rng.normal(0, 0.01, 3)
    q = np.array([1.0, *rng.normal(0, 0.003, 3)])
    x[3:7] = q / np.linalg.norm(q)
    x[7:10] = rng.normal(0, 0.004, 3)
    x[10:13] = rng.normal(0, 0.001, 3)
    th, ph, rho = rng.uniform(-0.3, 0.3, N), rng.uniform(-0.2, 0.2, N), 1 / rng.uniform(3, 12, N)
    anchors = rng.uniform(-0.2, 0.2, (N, 3))
    q1_angles(anchors, matched, th, ph)
    sd = np.zeros(n)
    sd[0:3], sd[3:7], sd[7:10], sd[10:13] = 0.02 * cam_sd, 0.005 * cam_sd, 0.01, 0.003
    for i in range(N):
        o = offs[i]
        if types[i]:
            x[o:o + 3] = [rng.uniform(-1.5, 1.5), rng.uniform(-1, 1), rng.uniform(4, 10)]
            sd[o:o + 3] = 0.002
        else:
            x[o:o + 3] = anchors[i]
            x[o + 3:o + 6] = th[i], ph[i], rho[i]
            sd[o:o + 6] = [0.002] * 3 + [0.0008] * 2 + [0.06 * rho[i]]
    U = rng.normal(0, 1.0, (n, 6)) * (0.3 * sd)[:, None]
    P = np.diag(sd ** 2) + U @ U.T
    P = np.asfortranarray(0.5 * (P + P.T))
    h, vis = NP.predict_h(CAM9, x, types)
    assert vis[matched].all()
    z = h + rng.normal(0, 0.4, (N, 2))
    k = np.arange(m)
    out1 = (rng.random(m) < outliers) & (k > 0) & (k < m - 1)
    out2 = (rng.random(m) < gross) & (k > 0) & (k < m - 1) & ~out1
    for sel, lo, hi in ((out1, 3, 15), (out2, 40, 80)):
        j = matched[sel]
        z[j] += rng.choice([-1.0, 1.0], (j.size, 2)) * rng.uniform(lo, hi, (j.size, 2))
    ic = np.zeros(N, bool)
    ic[matched] = True
    out = dict(types=types, x=x, P=P, z=z, ic=ic, matched=matched, offs=offs)
    for v in out.values():
        v.flags.writeable = False
    return out


def load(f, sc, b=0, ic=None):
    f.upload_state(sc["x"], sc["P"], feat_types=sc["types"], b=b, prior=True)
    f.predict_measurements()
    f.set_matches(sc["z"], (sc["ic"] if ic is None else ic).astype(np.uint8), b=b)


def device_supports(f, m):
    """every hypothesis' support and mask from one deduplicated sweep over the ids 0 .. m-1 (B = 1)"""
    key, _, pairs = f.support_sweep(np.arange(m, dtype=np.int32))
    assert pairs == m * m
    masks = np.array([f.sweep_mask(t)[:m] for t in range(m)])
    return masks.sum(axis=1), masks, key


def float64_check(f, sc, masks, q1, std_z):
    """every hypothesis' mask against float64 under the band rule, from the device's h, Hc, Hf"""
    fg = f.features()
    Hc, Hf = f.H_sparse()
    mt = sc["matched"]
    for t, p in enumerate(mt):
        res, *_ = support_reference(sc["x"], sc["P"], sc["offs"], Hc, Hf, fg["h"], sc["z"], p, mt, q1)
        band_check(masks[t], res, std_z, f"hypothesis {t}")


def check_select(f, res, exp, masks, matched, what=""):
    assert {k: res[k] for k in exp} == exp, (what, res, exp)
    if exp["winner"] >= 0:
        li = f.features()["li"]
        t = draw_t(f._u[exp["winner"]], len(matched))
        assert np.array_equal(li[matched], masks[t]), what


def run_select(f, u):
    f._u = np.asarray(u, np.float64)
    return f.ransac_hypotheses(f._u)


# ---- 1. support geometry -------------------------------------------------------------------------------------------------------------
# name: (N, m, cartesian, Q1, std_z).  N is kept close to m so that the matches reach the last 32-bit mask word of the handle.
GEOM = {"m1": (4, 1, 1, True, 1.0), "m31": (40, 31, 3, False, 0.6), "m32": (36, 32, 2, True, 1.7), "m33": (45, 33, 4, False, 1.0),
        "m63": (64, 63, 1, True, 0.6), "m64": (90, 64, 5, False, 1.7), "m65": (90, 65, 6, True, 1.0), "m127": (128, 127, 0, False, 1.0),
        "m128": (150, 128, 7, True, 1.7), "m129": (140, 129, 3, False, 0.6), "N256": (256, 198, 9, True, 1.0),
        "N257": (257, 200, 9, False, 1.7), "N1024": (1024, 700, 20, True, 1.7), "N1025": (1025, 900, 30, False, 1.0),
        "N1100": (1100, 1000, 25, True, 0.6)}


def test_geometry_cases_cover_the_edges():
    ms = [v[1] for v in GEOM.values()]
    assert {k % 6 for k in ms} == set(range(6))
    assert {v[3] for v in GEOM.values()} == {True, False} and {v[4] for v in GEOM.values()} == {0.6, 1.0, 1.7}
    Ns = {v[0] for v in GEOM.values()}
    assert {256, 257, 1024, 1025, 1100} <= Ns


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(GEOM))
def test_support_geometry(case):
    """Every hypothesis' support and mask against float64; the frame path's counters and li against select_reference driven by the
    device's supports; the launch profile of the set-up path (fused k_ransac_compact_hyp for N <= 256, else k_ransac_compact +
    k_ransac_hyp)."""
    N, m, nc, q1, std_z = GEOM[case]
    sc = geom_scene(N, m, nc)
    assert (sc["types"] == 1).sum() == nc and (nc > 0 or not np.array_equal(sc["matched"], np.arange(m)))  # offsets or id_list not the identity
    f = capi.Filter(CAM9, N, quirks=quirks(q1), std_z=std_z)
    try:
        load(f, sc)
        u = np.random.default_rng([N, 42]).random(700)
        f.profile(True)
        f.profile_read()
        res = run_select(f, u)
        prof = f.profile_read()
        f.profile(False)
        fused = N <= 256
        assert ("k_ransac_compact_hyp" in prof) == fused and ("k_ransac_compact" in prof) == (not fused), prof
        assert ("k_ransac_hyp" in prof) == (not fused)
        li = f.features()["li"]
        sup, masks, _ = device_supports(f, m)
        float64_check(f, sc, masks, q1, std_z)
        assert res["num_ic"] == m
        exp = select_reference(sup, m, u)
        f._u = u
        check_select(f, res, exp, masks, sc["matched"], case)
        assert np.array_equal(li, f.features()["li"])
        if m > 1:
            assert len(set(sup.tolist())) > 1, "supports must vary between hypotheses"
    finally:
        f.close()


# ---- 2. planted decisions ------------------------------------------------------------------------------------------------------------
HALF_PI = math.pi / 2
ANGLES = ([k * HALF_PI + s * 1e-6 for k in (-3, -2, -1, 0, 1, 2, 3, 4) for s in (1, -1)]
          + [k * HALF_PI + s * 1e-6 for k in (60000, -60000, 60001, -60003) for s in (1, -1)]
          + [1e5 - 1, 1e5 + 1, -1e5 + 1, -1e5 - 1])  # either side of sincos_fast's switch to the library sincos


@functools.lru_cache(maxsize=2)
def planted_scene(q1):
    """64 matched inverse-depth features; P block-diagonal (camera block, tiny diagonal feature blocks), so hypothesis 0 moves the camera
    and leaves every other feature's rows of x_i bitwise equal to x.  Probes 45..63: Q1 "angles" at k pi/2 +- 1e-6 and |a| = 1e5 +- 1
    (under Q1 they sit in the stacked positions of matches 30..42, otherwise in the probes' own angle rows), four image corners, and a
    point behind the hypothesised camera.  Each probe's z lies std_z (1 +- 1e-7) from its float64 re-projection, alternately inside and
    outside.  Returns dict with the inputs, the probes and their intended decisions."""
    std_z = 1.7 if q1 else 0.6
    rng = np.random.default_rng([int(q1), 43])
    N = m = 64
    types = np.zeros(N, np.int32)
    offs, _, n = layout(types)
    x = np.zeros(n)
    x[0:3] = rng.normal(0, 0.01, 3)
    q = np.array([1.0, *rng.normal(0, 0.003, 3)])
    x[3:7] = q / np.linalg.norm(q)
    th, ph, rho = rng.uniform(-0.3, 0.3, N), rng.uniform(-0.2, 0.2, N), 1 / rng.uniform(3, 12, N)
    anchors = rng.uniform(-0.2, 0.2, (N, 3))
    q1_angles(anchors, np.arange(N), th, ph)
    probes = list(range(45, 64))
    pairs = [(ANGLES[2 * k], ANGLES[2 * k + 1]) for k in range(len(ANGLES) // 2)]
    kinds = ["angles"] * len(pairs) + ["corner"] * 4 + ["behind"]
    assert len(kinds) == len(probes)
    corners = [(2.5, 2.5), (COLS - 2.5, 3.0), (3.0, ROWS - 2.5), (COLS - 3.0, ROWS - 3.0)]
    R = NP.q2r(x[3:7])
    k1, k2, _, _, Cx, Cy, fo, dx, dy = CAM9
    stacked = anchors.reshape(-1)
    for c, kind in zip(probes, kinds):
        if kind == "angles":
            a0, a1 = pairs[c - probes[0]]
            th[c], ph[c] = a0, a1
            if q1:
                stacked[2 * c], stacked[2 * c + 1] = a0, a1
            d = np.array([rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), 1.0]) * rng.uniform(3, 8)
        elif kind == "corner":
            uv = undistort(CAM9, np.array(corners[c - probes[0] - len(pairs)]))
            d = np.array([(uv[0] - Cx) * dx / fo, (uv[1] - Cy) * dy / fo, 1.0]) * rng.uniform(3, 8)
        else:
            d = np.array([0.3, -0.2, -4.0])
        a0, a1 = (stacked[2 * c], stacked[2 * c + 1]) if q1 else (th[c], ph[c])
        mi = np.array([np.cos(a1) * np.sin(a0), -np.sin(a1), np.cos(a1) * np.cos(a0)])
        rho[c] = 0.2
        anchors[c] = x[0:3] + (R @ d - mi) / rho[c]  # (r - x_c) rho + m = R d
    anchors = stacked.reshape(N, 3)
    for i in range(N):
        o = offs[i]
        x[o:o + 3] = anchors[i]
        x[o + 3:o + 6] = th[i], ph[i], rho[i]
    P = np.zeros((n, n), order="F")
    C = rng.normal(0, 1, (13, 13)) * 0.3
    sdc = np.array([0.02] * 3 + [0.005] * 4 + [0.01] * 3 + [0.003] * 3)
    P[:13, :13] = (C @ C.T + np.eye(13)) * sdc[:, None] * sdc[None, :]
    for i in range(N):
        o = offs[i]
        P[o:o + 6, o:o + 6] = np.diag(np.array([0.002] * 3 + [0.0008] * 2 + [0.06 * rho[i]]) ** 2)
    h, vis = NP.predict_h(CAM9, x, types)
    assert vis[0]
    Hc, Hf = np.zeros((N, 2, 7)), np.zeros((N, 2, 6))
    Hd = NP.jacobian_H(CAM9, x, types, 0, h[0])
    Hc[0], Hf[0] = Hd[:, :7], Hd[:, 13:19]
    z = h + rng.normal(0, 0.4, (N, 2))
    z[0] = h[0] + np.array([0.6, -0.3])
    ids = np.arange(N)
    res, hd, hc, xi = support_reference(x, P, offs, Hc, Hf, h, z, 0, ids, q1)
    inside = np.zeros(N, bool)
    for k, c in enumerate(probes):
        inside[c] = k % 2 == 0
        psi = rng.uniform(0, 2 * math.pi)
        z[c] = hd[c] + std_z * (1 + (-1e-7 if inside[c] else 1e-7)) * np.array([math.cos(psi), math.sin(psi)])
    out = dict(types=types, x=x, P=P, z=z, ic=np.ones(N, bool), matched=ids, offs=offs, h=h, Hc=Hc, Hf=Hf, probes=np.array(probes),
               kinds=kinds, inside=inside, std_z=std_z, q1=q1, xi=xi)
    return out


@pytest.mark.parametrize("q1", [True, False], ids=["q1", "no-q1"])
def test_planted_residuals_clear_the_threshold(q1):
    """Every planted residual lies at least 1e-9 std_z from std_z on its intended side, with K from the explicit inverse and from a
    solve; the probes reach their edges (the angles the support uses are the planted values, the corner probes re-project within 4 px
    of the corners, the behind probe has hc_z < 0, yet its residual is inside)."""
    sc = planted_scene(q1)
    std_z, pr = sc["std_z"], sc["probes"]
    for inv in (True, False):
        res, hd, hc, xi = support_reference(sc["x"], sc["P"], sc["offs"], sc["Hc"], sc["Hf"], sc["h"], sc["z"], 0, sc["matched"], q1, inv=inv)
        assert (np.abs(res[pr] - std_z) >= 1e-9 * std_z).all()
        assert np.array_equal(res[pr] < std_z, sc["inside"][pr])
    assert not np.array_equal(xi[:7], sc["x"][:7]) and np.array_equal(xi[19:], sc["x"][19:])  # only the camera and feature 0 move
    riv = xi[13:].reshape(-1, 6)[:, :3].reshape(-1)
    used = [(riv[2 * c], riv[2 * c + 1]) if q1 else (xi[13 + 6 * c + 3], xi[13 + 6 * c + 4]) for c in pr]
    na = len(ANGLES) // 2
    assert [a for pair in used[:na] for a in pair] == ANGLES
    for k, c in enumerate(pr[na:na + 4]):
        corner = np.array([[2.5, 2.5], [COLS - 2.5, 3.0], [3.0, ROWS - 2.5], [COLS - 3.0, ROWS - 3.0]][k])
        assert np.abs(hd[c] - corner).max() < 4
    assert hc[2, pr[-1]] < 0 and sc["inside"][pr[-1]]


@pytest.mark.gpu
@pytest.mark.parametrize("q1", [True, False], ids=["q1", "no-q1"])
def test_planted_decisions(q1):
    """The probes' decisions under hypothesis 0 are exact; every other decision of that hypothesis is held to the band rule."""
    sc = planted_scene(q1)
    f = capi.Filter(CAM9, 64, quirks=quirks(q1), std_z=sc["std_z"])
    try:
        load(f, sc)
        key, mask, pairs = f.support_sweep(np.array([0], np.int32))
        assert pairs == 64
        got = f.sweep_mask(0)[:64]
        pr = sc["probes"]
        bad = [(int(c), k) for c, k in zip(pr, sc["kinds"]) if got[c] != sc["inside"][c]]
        assert not bad, f"planted decisions differ: {bad}"
        res, *_ = support_reference(sc["x"], sc["P"], sc["offs"], sc["Hc"], sc["Hf"], sc["h"], sc["z"], 0, sc["matched"], q1)
        band_check(got, res, sc["std_z"], "hypothesis 0")
        assert key >> 32 == got.sum()
    finally:
        f.close()


# ---- 3. selection --------------------------------------------------------------------------------------------------------------------
SEL = (160, 150, 6)  # N, nIC, cartesian


def sel_scene():
    return geom_scene(*SEL, seed=1, outliers=0.2, gross=0.15)


def selection_draws(sup, nic, p, rng):
    """{name: u01} built against the supports: where the first record falls, records inside one chunk, records past the current
    index, exhausted draws on both paths of k_select, ties, u = 0 / nextafter(1, 0) / 1."""
    zero = [t for t in range(nic) if sup[t] == 0]
    pos = sorted({int(s) for s in sup if s > 0})
    by = {s: [t for t in range(nic) if sup[t] == s] for s in pos}
    uo = lambda t: (t + 0.5) / nic  # noqa: E731
    zeros = lambda k: [uo(zero[i % len(zero)]) for i in range(k)]  # noqa: E731
    tail = list(rng.random(3000))
    smax = pos[-1]
    out = {}
    for k in (0, 31, 32, 33):
        out[f"first-record-at-{k}"] = zeros(k) + [uo(by[pos[len(pos) // 2]][0])] + tail
    ladder = [uo(by[s][0]) for s in pos[:6]]
    out["records-in-one-chunk"] = zeros(3) + [ladder[0]] + zeros(2) + ladder[1:3] + zeros(5) + ladder[3:6] + tail
    nh = n_hyp_of(smax, nic, p)
    out["record-n_hyp-below-index"] = zeros(nh + 20) + [uo(by[smax][0])] + tail
    out["record-n_hyp-equal-index"] = zeros(nh) + [uo(by[smax][0])] + tail
    tie = [s for s in pos if len(by[s]) > 1][-1]
    out["equal-support-later"] = [uo(by[tie][0]), uo(by[tie][1])] + zeros(40) + [uo(by[tie][-1])] + zeros(3000)
    out["u0-and-below-1"] = [0.0, float(np.nextafter(1.0, 0.0))] + zeros(5) + tail
    out["u1-resolved"] = zeros(5) + [1.0] + tail
    out["u1-direct"] = zeros(9000) + [1.0] + zeros(100)
    for k in (8191, 8192, 8193, 10000):
        out[f"record-at-{k}"] = zeros(k) + [uo(by[pos[0]][0])] + zeros(50)
    return out


@pytest.mark.gpu
def test_selection():
    """k_ransac_select against select_reference on draws constructed against the device's supports (themselves checked against
    float64): records at the chunk edges 31 / 32 / 33 and past the resolved draws 8192, records inside a chunk, a record whose n_hyp lies
    below / at the current index, equal supports later, u = 0, nextafter(1, 0) and 1.0 on both paths, exhausted draws at every block edge,
    nIC = 0, p_spurious_free in {0.5, 0.99, 0.999} and n_hyp_initial in {0, 1, 50, 64, 20000}."""
    sc = sel_scene()
    N, nic, _ = SEL
    mt = sc["matched"]
    handles = {}
    try:
        for p in (0.5, 0.99, 0.999):
            for n0 in (0, 1, 50, 64, 20000):
                handles[p, n0] = f = capi.Filter(CAM9, N, quirks=quirks(False), p_spurious_free=p, n_hyp_initial=n0)
                load(f, sc)
        f0 = handles[0.99, 1000] = capi.Filter(CAM9, N, quirks=quirks(False))
        load(f0, sc)
        sup, masks, _ = device_supports(f0, nic)
        float64_check(f0, sc, masks, False, 1.0)
        assert (sup == 0).sum() >= 3 and len(set(sup[sup > 0].tolist())) >= 6 and sup[0] > 0 and sup[-1] > 0
        rng = np.random.default_rng(44)
        reached = set()
        for (p, n0), f in handles.items():
            for name, u in selection_draws(sup, nic, p, rng).items():
                res = run_select(f, u)
                exp = select_reference(sup, nic, u, p, n0)
                check_select(f, res, exp, masks, mt, f"{name} p = {p} n_hyp0 = {n0}")
                if n0 == 1000 or n0 == 20000:
                    w = exp["winner"]
                    reached.add((name, w))
        for k in (0, 31, 32, 33, 8191, 8192, 8193, 10000):
            assert any(w == k for nm, w in reached if nm.endswith(f"-at-{k}") or nm == f"first-record-at-{k}"), k
        assert ("u1-direct", 9000) in reached and ("u1-resolved", 5) in reached
        # exhausted draws at every block edge of k_select (no record: every draw has support 0), and a loop ending at a chunk end
        zero = [t for t in range(nic) if sup[t] == 0]
        f = handles[0.99, 20000]
        for n_u in (1, 31, 32, 33, 2047, 2048, 2049, 8191, 8192, 8193, 12000):
            u = [(zero[i % len(zero)] + 0.5) / nic for i in range(n_u)]
            res = run_select(f, u)
            assert {k: res[k] for k in ("status", "hyp_run", "best_support", "winner")} == dict(status=3, hyp_run=n_u, best_support=0, winner=-1)
        res = run_select(handles[0.99, 64], [(zero[0] + 0.5) / nic] * 100)
        assert (res["status"], res["hyp_run"], res["n_hyp"]) == (0, 64, 64)
        with pytest.raises(capi.RslamError):
            f.ransac_hypotheses(np.zeros(0))
        # nIC = 0 (Q9)
        f.set_matches(sc["z"], np.zeros(N, np.uint8))
        res = run_select(f, [0.5] * 10)
        assert {k: res[k] for k in ("status", "hyp_run", "best_support", "n_hyp", "num_ic", "winner")} == dict(
            status=1, hyp_run=0, best_support=0, n_hyp=20000, num_ic=0, winner=-1)
    finally:
        for f in handles.values():
            f.close()


# ---- 4. n_hyp rounding ---------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def uniform_scene(N=1000):
    """Zero camera rows and columns in P, no cross-covariances, feature variances of 1e-14: every hypothesis leaves the camera where it
    is, so every hypothesis scores the same support, the number of matches planted at 0.5 std_z (the others at 2 std_z)."""
    rng = np.random.default_rng(45)
    types = np.zeros(N, np.int32)
    offs, _, n = layout(types)
    x = np.zeros(n)
    x[3] = 1.0
    for i in range(N):
        o = offs[i]
        x[o:o + 3] = rng.uniform(-0.2, 0.2, 3)
        x[o + 3:o + 6] = rng.uniform(-0.3, 0.3), rng.uniform(-0.2, 0.2), 1 / rng.uniform(3, 12)
    P = np.zeros((n, n), order="F")
    P[np.arange(13, n), np.arange(13, n)] = 1e-14
    h, vis = NP.predict_h(CAM9, x, types)
    assert vis.all()
    return types, x, P, h


def uniform_matches(h, s, nic, N):
    z = h + np.array([2.0, 0.0])
    z[:s] = h[:s] + np.array([0.0, 0.5])
    ic = np.zeros(N, np.uint8)
    ic[:nic] = 1
    return z, ic


@pytest.mark.gpu
@pytest.mark.parametrize("p", sorted(NHYP_PINS))
def test_n_hyp_rounding(p):
    """The device's n_hyp on members of the near-integer families of test_n_hyp_near_integer_scan (nIC <= 1000), on support = nIC
    (n_hyp = 0) and on ordinary ratios, equals ceil of libm's ratio; hyp_run follows."""
    types, x, P, h = uniform_scene()
    N = len(types)
    fams = NHYP_PINS[p][2]
    cases = [(a * k, b * k) for a, b in fams for k in (1, 10, 100) if b * k <= N] + [(10, 10), (1000, 1000), (500, 1000), (1, 7), (37, 40)]
    f = capi.Filter(CAM9, N, quirks=quirks(False), p_spurious_free=p)
    try:
        f.upload_state(x, P, feat_types=types, prior=True)
        f.predict_measurements()
        for s, nic in cases:
            z, ic = uniform_matches(h, s, nic, N)
            f.set_matches(z, ic)
            u = [0.5] * 64
            res = f.ransac_hypotheses(u)
            exp = select_reference([s] * nic, nic, u, p)
            assert {k: res[k] for k in exp} == exp, (s, nic, res, exp)
        assert n_hyp_of(10, 10, p) == 0
    finally:
        f.close()


# ---- 5. batch ------------------------------------------------------------------------------------------------------------------------
BATCH = [(10, 0), (3, 1), (8, 6), (70, 65), (260, 257), (1030, 1025)]  # (N, nIC)


@pytest.mark.gpu
def test_batch_members_equal_singles_and_the_reference():
    """One rslam_ransac_hypotheses call on six heterogeneous members (nIC = 0, 1, 6, 65, 257, 1025): each member's counters and li equal
    the same filter run alone (B = 1) bit for bit, and select_reference over that filter's supports."""
    Nmax = max(N for N, _ in BATCH)
    scenes = [geom_scene(N, max(nic, 1), 0, seed=2) for N, nic in BATCH]
    ics = [sc["ic"] if nic else np.zeros(N, bool) for sc, (N, nic) in zip(scenes, BATCH)]
    rng = np.random.default_rng(46)
    U = rng.random((len(BATCH), 900))
    bat = capi.Filter(CAM9, Nmax, batch=len(BATCH), std_z=1.7)
    try:
        for b, sc in enumerate(scenes):
            bat.upload_state(sc["x"], sc["P"], feat_types=sc["types"], b=b, prior=True)
        bat.predict_measurements()
        for b, sc in enumerate(scenes):
            bat.set_matches(sc["z"], ics[b].astype(np.uint8), b=b)
        bat.ransac_hypotheses(U)
        for b, (sc, (N, nic)) in enumerate(zip(scenes, BATCH)):
            one = capi.Filter(CAM9, Nmax, std_z=1.7)
            try:
                load(one, sc, ic=ics[b])
                r1 = run_select(one, U[b])
                rb = bat.ransac_result(b)
                assert rb == r1, (b, rb, r1)
                li1 = one.features()["li"]
                assert np.array_equal(bat.features(b)["li"], li1), b
                if nic == 0:
                    assert r1["status"] == 1
                    continue
                sup, masks, _ = device_supports(one, nic)
                exp = select_reference(sup, nic, U[b])
                check_select(one, r1, exp, masks, sc["matched"], f"member {b}")
            finally:
                one.close()
    finally:
        bat.close()


# ---- 6. sweep ------------------------------------------------------------------------------------------------------------------------
def sweep_expect(sup, hyp, begin, end, m_lo, m_hi, m, dedupe):
    key, valid = 0, []
    for i in range(begin, end):
        t = int(hyp[i])
        if m_lo <= t < min(len(sup), m_hi):
            valid.append(t)
            key = max(key, (int(sup[t]) << 32) | (0xFFFFFFFF - i))
    pairs = (len(set(valid)) if dedupe else len(valid)) * m
    return key, pairs


@pytest.mark.gpu
def test_sweep():
    """rslam_support_sweep's key, mask and pair count against the device's verified supports: id lists with duplicates and ids >= nIC
    (ignored), hyp_begin > 0, host and device lists, match ranges that cut a 6-hypothesis batch and a 64-match tile, ties (the lowest id
    wins), an empty selection (key 0), dedupe on and off giving the same keys and masks."""
    import torch

    sc = sel_scene()
    N, nic, _ = SEL
    fs = {d: capi.Filter(CAM9, N, quirks=quirks(False), dedupe=d) for d in (True, False)}
    try:
        for f in fs.values():
            load(f, sc)
        sup, masks, _ = device_supports(fs[True], nic)
        float64_check(fs[True], sc, masks, False, 1.0)
        smax = int(sup.max())
        tops = np.flatnonzero(sup == smax)
        tie = [s for s in sorted(set(sup.tolist())) if (sup == s).sum() > 1][-1]
        ties = np.flatnonzero(sup == tie)
        rng = np.random.default_rng(47)
        base = rng.integers(0, nic + 40, 300).astype(np.int32)  # duplicates and ids >= nIC
        lists = {
            "dup-and-out-of-range": (base, 7, 290, 0, 2**31 - 1),
            "match-range-cuts-batch-and-tile": (base, 0, 300, 4, 71),
            "top-twice-lowest-id-wins": (np.array([nic + 3, int(tops[0]), 5, int(tops[0]), int(tops[-1])], np.int32), 0, 5, 0, 2**31 - 1),
            "equal-supports-distinct-ids": (np.array([int(ties[1]), int(ties[0]), nic, int(ties[1])], np.int32), 0, 4, 0, 2**31 - 1),
            "begin-past-the-best": (np.array([int(tops[0])] + [int(t) for t in ties], np.int32), 1, 1 + len(ties), 0, 2**31 - 1),
            "empty": (np.array([nic, nic + 1, nic + 5], np.int32), 0, 3, 0, 2**31 - 1),
            "empty-range": (base, 10, 10, 0, 2**31 - 1),
        }
        for name, (hyp, b, e, mlo, mhi) in lists.items():
            got = {}
            for d, f in fs.items():
                exp_key, exp_pairs = sweep_expect(sup, hyp, b, e, mlo, mhi, nic, d)
                key, mask, pairs = f.support_sweep(hyp, begin=b, end=e, match_begin=mlo, match_end=mhi)
                assert (key, pairs) == (exp_key, exp_pairs), (name, d, capi.decode_key(key), capi.decode_key(exp_key), pairs, exp_pairs)
                if key:
                    assert np.array_equal(mask[:nic], masks[int(hyp[capi.decode_key(key)[1]])]), (name, d)
                else:
                    assert not mask[:nic].any(), (name, d)
                dh = torch.from_numpy(np.ascontiguousarray(hyp)).cuda()
                kd, maskd, pd = f.support_sweep(dh.data_ptr(), n_hyp=hyp.size, begin=b, end=e, match_begin=mlo, match_end=mhi)
                assert (kd, pd) == (key, pairs) and np.array_equal(maskd, mask), (name, d, "device list")
                got[d] = (key, mask[:nic].copy())
            assert got[True][0] == got[False][0] and np.array_equal(got[True][1], got[False][1]), name
        k = capi.decode_key(fs[True].support_sweep(lists["top-twice-lowest-id-wins"][0])[0])
        assert k == (smax, 1)
        k = capi.decode_key(fs[True].support_sweep(lists["equal-supports-distinct-ids"][0])[0])
        assert k == (tie, 0)
    finally:
        for f in fs.values():
            f.close()
