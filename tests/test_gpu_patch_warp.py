"""The predicted-appearance warp -- k_pred_patch_setup and k_pred_patch, Tracking::pred_patch_fc (src/Tracking.cpp:164-278) on the
device -- against an exact remap and a float64 reference, at the edges where it can go wrong.

Inputs are planted through the C ABI: the prior state (rslam_upload_state, which also fixes the feature types and so the stale XYZ_w
of quirk Q3), the initial patches and poses (rslam_upload_feature_init), then rslam_predict_measurements with the warp on.  h is
whatever k_predict computes from the planted state.

Why the reference can be exact.  The sampling half of the warp is exact arithmetic: taps are integers 0..255 and the bilinear weights
are products of multiples of 1/32, so every output is k / 1024 and every float operation of tap * w00 + ... is exact, in any order and
with or without FMA contraction.  The only rounding is in the geometry, up to the cast of a map coordinate to float and its 1/32-px
quantisation.  On a dyadic pinhole camera (k1 = k2 = 0, f / dx = 256) undistort and distort are identities in floating point, K and K^-1
are dyadic, and for signed permutations (and dyadic shears) as initial rotations, axis translations with the plane normal on the optical
axis, and dyadic initial pixels, every operation of the geometry is exact as well.  There the device must equal, bit for bit, an
integer remap sum(tap * wy * wx) / 1024 of the map coordinates computed in rational arithmetic (`exact_maps`).

On the real, distorted camera the reference is np_oracle.pred_patch_maps (float64) followed by the same integer remap: a pixel may
take either of two values only where float32(m - 1e-9 px) and float32(m + 1e-9 px) quantise differently (the band), and window
truncations and gates are kept more than 1e-9 from their thresholds, which the CPU tests assert."""
import functools
import math
from fractions import Fraction as Fr

import numpy as np
import pytest

from oracle import np_oracle as NP
from ransac_slam_b200 import capi, synth
from tests import test_gpu_track_kernels as TK

CAM_D = np.array([0.0, 0.0, 240, 320, 160.0, 120.0, 1.0, 2.0**-8, 2.0**-8])  # dyadic pinhole: f / dx = 256
CAM_R = synth.Camera().as9()  # the distorted camera of the synthetic scenes
ROWS, COLS = 240, 320
HP = 6
BAND = 1e-9  # px

I3 = np.eye(3)
ROT90 = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1.0]])
ROT180 = np.diag([-1.0, -1.0, 1.0])
MIRROR = np.diag([-1.0, 1.0, 1.0])  # a reflection (det = -1): R_wc_when_initialized need not be a rotation
SHEAR = np.array([[1, 0, 0], [0, 1, 0], [0, 0.5, 1.0]])  # dyadic, not orthonormal: a vanishing line crosses the window


# ---- exact reference ------------------------------------------------------------------------------------------------------------
def _mm(A, B):
    return [[sum(A[i][k] * B[k][j] for k in range(len(B))) for j in range(len(B[0]))] for i in range(len(A))]


def _mv(A, v):
    return [sum(A[i][k] * v[k] for k in range(len(v))) for i in range(len(A))]


def _inv(A):
    n = len(A)
    M = [list(A[i]) + [Fr(int(i == j)) for j in range(n)] for i in range(n)]
    for c in range(n):
        p = next(r for r in range(c, n) if M[r][c] != 0)
        M[c], M[p] = M[p], M[c]
        piv = M[c][c]
        M[c] = [v / piv for v in M[c]]
        for r in range(n):
            if r != c and M[r][c] != 0:
                fac = M[r][c]
                M[r] = [a - fac * b for a, b in zip(M[r], M[c])]
    return [row[n:] for row in M]


def _esqrt(q):
    """the square root of a rational that has an exact one (asserted): the cases are built so that the normalisations are exact"""
    a, b = math.isqrt(q.numerator), math.isqrt(q.denominator)
    assert a * a == q.numerator and b * b == q.denominator, f"sqrt({q}) is not exact"
    return Fr(a, b)


def _homog(R, r):  # [R 0; 0 1] [I r; 0 1] (quirk Q12)
    Rr = _mv(R, r)
    return [R[0] + [Rr[0]], R[1] + [Rr[1]], R[2] + [Rr[2]], [Fr(0), Fr(0), Fr(0), Fr(1)]]


def _q2r(q):
    r, x, y, z = (Fr(float(v)) for v in q)
    return [[r * r + x * x - y * y - z * z, 2 * (x * y - r * z), 2 * (z * x + r * y)],
            [2 * (x * y + r * z), r * r - x * x + y * y - z * z, 2 * (y * z - r * x)],
            [2 * (z * x - r * y), 2 * (y * z + r * x), r * r - x * x - y * y + z * z]]


def exact_xyz_w(x, types, i):
    """np_oracle.xyz_w_for_warp in rational arithmetic; the inverse-depth features of the exact cases have theta = phi = 0"""
    last = [k for k in range(i + 1) if types[k] == 0]
    if not last:
        return [Fr(0)] * 3
    offs, _, _ = TK.layout(types)
    y = x[offs[last[-1]]:offs[last[-1]] + 6]
    assert y[3] == 0 and y[4] == 0 and Fr(1.0 / y[5]) == 1 / Fr(y[5])
    return [Fr(y[0]), Fr(y[1]), Fr(y[2]) + 1 / Fr(y[5])]


def exact_maps(cam, x, h, X, r_init, R_init, uvf):
    """pred_patch_fc's geometry in rational arithmetic on a dyadic pinhole camera.  Returns (xs, ys, ok, maps) as np_oracle.pred_patch_maps,
    maps[r][c] = (mx, my) as Fractions, or None where the pixel lies on the homography's vanishing line (w2 == 0: the float pipeline
    gives NaN)."""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = (Fr(float(v)) for v in cam)
    assert k1 == 0 and k2 == 0 and dx == dy
    hx, hy = Fr(float(h[0])), Fr(float(h[1]))
    if not (HP < hx < nCols - HP and HP < hy < nRows - HP):
        return 0, 0, -1, None
    fk = f / dx
    u0, v0 = Fr(float(uvf[0])), Fr(float(uvf[1]))
    R = [[Fr(float(v)) for v in row] for row in np.asarray(R_init, float).reshape(3, 3)]
    Hpfi = _inv(_homog(R, [Fr(float(v)) for v in r_init]))
    Hkk = _mm(Hpfi, _homog(_q2r(x[3:7]), [Fr(float(v)) for v in x[0:3]]))
    R12 = [row[:3] for row in Hkk[:3]]
    t = [Hkk[a][3] for a in range(3)]
    if any(t):
        n1 = [u0 - Cx, v0 - Cy, -fk]
        nn = _esqrt(sum(v * v for v in n1))
        n = [v / nn for v in n1]
        nt4 = _mv(Hkk, [hx - Cx, hy - Cy, -fk, Fr(1)])
        nt = [v / nt4[3] for v in nt4[:3]]
        ntn = _esqrt(sum(v * v for v in nt))
        ns = [a + b / ntn for a, b in zip(n, nt)]
        nsn = _esqrt(sum(v * v for v in ns))
        n = [v / nsn for v in ns]
        Xk = _mv(Hpfi, list(X) + [Fr(1)])
        d = -sum(n[a] * Xk[a] / Xk[3] for a in range(3))
        M = [[R12[a][b] - t[a] * n[b] / d for b in range(3)] for a in range(3)]
    else:  # t n^T / d vanishes whatever n and d are (as long as they are finite, d != 0)
        M = R12
    K = [[fk, Fr(0), Cx], [Fr(0), fk, Cy], [Fr(0), Fr(0), Fr(1)]]
    Hm = _mm(_mm(K, M), _inv(K))
    c = _mv(_inv(Hm), [u0, v0, Fr(1)])
    c2u, c2v = c[0] / c[2], c[1] / c[2]
    xs, xe, ys, ye = int(c2u - HP), int(c2u + HP), int(c2v - HP), int(c2v + HP)  # int() truncates toward zero, like cv::Range
    if xe - xs != 2 * HP or ye - ys != 2 * HP:
        return xs, ys, 0, None
    maps = []
    for r in range(13):
        row = []
        for cc in range(13):
            p = _mv(Hm, [Fr(xs + cc), Fr(ys + r), Fr(1)])
            row.append(None if p[2] == 0 else (p[0] / p[2] - (u0 - 21), p[1] / p[2] - (v0 - 21)))
        maps.append(row)
    return xs, ys, 1, maps


def quantise(m):
    """cv::remap's fixed-point map: cvRound(32 * float(m)), round half to even (m float64 scalars or arrays)"""
    return np.rint(np.asarray(np.float32(m), np.float64) * 32).astype(np.int64)


def remap_q(p41, sx, sy):
    """the exact bilinear sample of the uint8 41 x 41 patch at quantised coordinates (int arrays), border value 0"""
    p = np.asarray(p41, np.int64)
    ix, iy, ax, ay = sx >> 5, sy >> 5, sx & 31, sy & 31

    def tap(yy, xx):
        ok = (xx >= 0) & (xx < 41) & (yy >= 0) & (yy < 41)
        return np.where(ok, p[np.clip(yy, 0, 40), np.clip(xx, 0, 40)], 0)

    k = tap(iy, ix) * (32 - ay) * (32 - ax) + tap(iy, ix + 1) * (32 - ay) * ax + tap(iy + 1, ix) * ay * (32 - ax) + tap(iy + 1, ix + 1) * ay * ax
    return k / 1024.0


def exact_patch(p41, ok, maps):
    out = np.zeros((13, 13))
    if ok != 1:
        return out
    for r in range(13):
        for c in range(13):
            if maps[r][c] is not None:  # NaN map coordinate: out of range, the border value 0 (cvRound(NaN) is INT_MIN on x86)
                mx, my = maps[r][c]
                out[r, c] = remap_q(p41, quantise(float(mx)), quantise(float(my)))
    return out


def band_values(p41, mapx, mapy):
    """per pixel the values the remap can take when each float64 map coordinate may be off by BAND: (lo, hi, in_band)"""
    nan = np.isnan(mapx) | np.isnan(mapy)
    mx, my = np.where(nan, -1e6, mapx), np.where(nan, -1e6, mapy)
    qx = [quantise(mx - BAND), quantise(mx + BAND)]
    qy = [quantise(my - BAND), quantise(my + BAND)]
    vals = np.stack([remap_q(p41, a, b) for a in qx for b in qy])
    return vals.min(0), vals.max(0), (qx[0] != qx[1]) | (qy[0] != qy[1]), vals


# ---- planted maps on the dyadic camera ------------------------------------------------------------------------------------------
def id_feat(X, rho=0.5):
    """an inverse-depth feature with theta = phi = 0 whose point is X (the anchor 1 / rho behind it on the optical axis direction)"""
    return 0, [X[0], X[1], X[2] - 1.0 / rho, 0.0, 0.0, rho]


def cart_feat(X):
    return 1, list(X)


BEHIND = (0, [0.0, 0.0, 0.0, math.pi, 0.0, 0.5])  # an inverse-depth feature pointing backwards: never predicted (has_h = 0)


def gate_X(h):
    """a point at depth 1 whose exact projection on the dyadic camera is h"""
    X = [(Fr(float(h[0])) - 160) / 256, (Fr(float(h[1])) - 120) / 256]
    assert all(Fr(float(v)) == v for v in X)
    return [float(X[0]), float(X[1]), 1.0]


def ofs(k):  # a sub-pixel offset k / 256 px
    return k / 256.0


def lattice_features():
    """(name, (type, params), r_init, R_init, uvf) of the exact filter, in list order (the order decides XYZ_w, quirk Q3)"""
    A = id_feat([0.0, 0.0, 2.0])  # straight ahead, h = (160, 120)
    F = []
    # quirk Q3: a cartesian feature ahead of every inverse-depth one uses XYZ_w = 0: d = 1, zoom-in x 2 (its own point would give 3/2)
    F.append(("q3-cartesian-first-zoom-in", cart_feat([0.0, 0.0, 1.0]), [0, 0, -1.0], I3, [160.0, 120.0]))
    F.append(("identity-subpixel", A, [0, 0, 0], I3, [100 + ofs(77), 80 + ofs(179)]))
    # quantisation ties: a map coordinate k + 1/2 in 1/32 px rounds to even, up (1/64, -3/64 offsets) or down (-1/64, 3/64)
    F.append(("ties-up-x-down-y", A, [0, 0, 0], I3, [100 + 1 / 64, 80 - 1 / 64]))
    F.append(("ties-down-x-up-y", A, [0, 0, 0], I3, [100 + 3 / 64, 80 - 3 / 64]))
    F.append(("ties-down-x-down-y", A, [0, 0, 0], I3, [100 - 1 / 64, 80 + 3 / 64]))
    F.append(("ties-up-x-up-y", A, [0, 0, 0], I3, [100 - 3 / 64, 80 + 1 / 64]))
    F.append(("rot90-ties-y", A, [0, 0, 0], ROT90, [100.25, 80.5 + 1 / 64]))
    F.append(("rot180-ties-x", A, [0, 0, 0], ROT180, [100.25 + 1 / 64, 80.5]))
    F.append(("mirror", A, [0, 0, 0], MIRROR, [90 + 1 / 64, 70.75]))
    # window truncation (quirk Q13): c2u - 6 in (-1, 0) gives a 12-wide window and the zero patch, c2u - 6 = 0 a 13-wide one
    F.append(("window-12-wide-x", A, [0, 0, 0], I3, [5.5, 80.0]))
    F.append(("window-12-wide-y", A, [0, 0, 0], I3, [80.0, 5.5]))
    F.append(("window-12-wide-x-negative", A, [0, 0, 0], I3, [-0.5, 80.0]))
    F.append(("window-at-0-x", A, [0, 0, 0], I3, [6.0, 80.0 + ofs(3)]))
    F.append(("window-at-0-y", A, [0, 0, 0], I3, [80.0 + ofs(5), 6.0]))
    F.append(("window-negative-coordinates", A, [0, 0, 0], I3, [3.0, 2.0]))
    # the shear's vanishing line v = 632 crosses row 8 of the window: w2 == 0, NaN map coordinates, border value 0
    F.append(("vanishing-line", A, [0, 0, 0], SHEAR, [160.0, 130680.0]))
    # zoom-out x 4 about the principal point (the plane normal on the optical axis): maps span -3 .. 45, taps outside on every side,
    # index 41 included
    F.append(("zoom-out-4", id_feat([0.0, 0.0, 3.5]), [0, 0, 1.5], I3, [160.0, 120.0]))
    # cartesian features after it (Q3: XYZ_w = (0, 0, 3.5)), translated sideways so that the map is off-centre by a sub-pixel amount:
    # taps -1 and 0 and 39 and 40 in one axis, 40 and 41 in the other; h = C - (tx, ty) keeps the plane normal on the axis
    for nm, tx, ty in (("zoom-out-4-offset-a", 5 / 1024, 7 / 1024), ("zoom-out-4-offset-b", 7 / 1024, 5 / 1024)):
        F.append((nm, cart_feat([-tx / 64, -ty / 64, 4.0]), [-tx, -ty, 1.5], I3, [160.0, 120.0]))
    # zoom-out x 2, then a cartesian feature behind it that zooms with its XYZ_w (d = 2: x 2) and not with its own point (d = 7)
    F.append(("zoom-out-2", id_feat([0.0, 0.0, 3.0]), [0, 0, 1.0], I3, [160.0, 120.0]))
    F.append(("q3-cartesian-after-inverse-depth", cart_feat([0.0, 0.0, 8.0]), [0, 0, 1.0], I3, [160.0, 120.0]))
    # the border gate of h (src/Tracking.cpp:174-175): exactly 6 and nCols / nRows - 6 are rejected, one float step inside accepted
    for nm, h in (("gate-x-6", (6.0, 120.0)), ("gate-x-6+", (6 + 2.0**-45, 120.0)), ("gate-x-314", (314.0, 120.0)),
                  ("gate-x-314-", (314 - 2.0**-44, 120.0)), ("gate-y-6", (160.0, 6.0)), ("gate-y-6+", (160.0, 6 + 2.0**-46)),
                  ("gate-y-234", (160.0, 234.0)), ("gate-y-234-", (160.0, 234 - 2.0**-45))):
        F.append((nm, id_feat(gate_X(h), rho=1.0), [0, 0, 0], I3, [100 + ofs(77), 80 + ofs(179)]))
    F.append(("not-predicted", BEHIND, [0, 0, 0], I3, [100.0, 80.0]))
    return F


def build_filter_state(feats, r_cur=(0.0, 0.0, 0.0)):
    types = np.array([t for _, (t, _), *_ in feats], np.int32)
    x = [*r_cur, 1.0, 0, 0, 0, 0, 0, 0, 0, 0, 0]
    for _, (_, p), *_ in feats:
        x += list(p)
    return types, np.array(x, float)


def patches41(seed, N):
    p = np.random.default_rng([seed, 41]).integers(1, 256, (N, 41, 41)).astype(np.uint8)
    p[:, 0, 0] = 200  # what a NaN coordinate would read if it were rounded to 0
    return p


def init_arrays(feats):
    r = np.array([np.asarray(fe[2], float) for fe in feats])
    R = np.array([np.asarray(fe[3], float).reshape(9) for fe in feats])
    uv = np.array([np.asarray(fe[4], float) for fe in feats])
    return r, R, uv


def expected_exact(cam, feats, types, x, p41):
    """(has_h, h, per feature (xs, ys, ok, maps) of exact_maps, expected patches)"""
    h, vis = NP.predict_h(cam, x, types)
    out = np.zeros((len(feats), 13, 13))
    geo = []
    for i, fe in enumerate(feats):
        if not vis[i]:
            geo.append(None)
            continue
        xs, ys, ok, maps = exact_maps(cam, x, h[i], exact_xyz_w(x, types, i), fe[2], fe[3], fe[4])
        geo.append((xs, ys, ok, maps))
        out[i] = exact_patch(p41[i], ok, maps)
    return vis, h, geo, out


@functools.lru_cache(maxsize=None)
def lattice_case():
    feats = lattice_features()
    types, x = build_filter_state(feats)
    p41 = patches41(1, len(feats))
    vis, h, geo, exp = expected_exact(CAM_D, feats, types, x, p41)
    return feats, types, x, p41, vis, h, geo, exp


def run_warp(f, b, types, x, p41, feats, prior_P=None):
    n = x.size
    f.upload_state(x, np.eye(n) * 1e-4 if prior_P is None else prior_P, feat_types=types, b=b, prior=True)
    r, R, uv = init_arrays(feats)
    f.upload_feature_init(p41, r, R, uv, b=b)


def assert_patches_equal(got, exp, names, what=""):
    bad = []
    for i, nm in enumerate(names):
        d = got[i].astype(np.float64) != exp[i]
        if d.any():
            r, c = np.argwhere(d)[0]
            bad.append(f"{nm}: {int(d.sum())} pixels, first ({r}, {c}) got {got[i][r, c]} want {exp[i][r, c]}")
    assert not bad, f"{what}: " + "; ".join(bad)


# ---- CPU: the planted cases reach their edges, and the references agree with the C++ oracle -------------------------------------
def test_lattice_cases_reach_their_edges():
    """Each exact case sits where its name says: gates exactly on / one step inside, the window widths, ties in both directions,
    taps outside the patch, the NaN row, the Q3 zooms; every map coordinate of an exact case is a float64 (so the device's value)."""
    feats, types, x, p41, vis, h, geo, exp = lattice_case()
    g = {fe[0]: (i, geo[i]) for i, fe in enumerate(feats)}
    assert not vis[g["not-predicted"][0]] and vis.sum() == len(feats) - 1
    for nm, axis, want in (("gate-x-6", 0, 6.0), ("gate-x-6+", 0, 6 + 2.0**-45), ("gate-x-314", 0, 314.0), ("gate-x-314-", 0, 314 - 2.0**-44),
                           ("gate-y-6", 1, 6.0), ("gate-y-6+", 1, 6 + 2.0**-46), ("gate-y-234", 1, 234.0), ("gate-y-234-", 1, 234 - 2.0**-45)):
        i, gi = g[nm]
        assert h[i][axis] == want, nm
        inside = nm.endswith(("+", "-"))
        assert (gi[2] == 1) == inside and (gi[2] == -1) == (not inside), nm
    for nm in ("window-12-wide-x", "window-12-wide-y", "window-12-wide-x-negative"):
        assert g[nm][1][2] == 0, nm
    assert g["window-at-0-x"][1][:3] == (0, 74, 1) and g["window-at-0-y"][1][:3] == (74, 0, 1)
    assert g["window-negative-coordinates"][1][:3] == (-3, -4, 1)
    ties = {"up": set(), "down": set()}
    taps = set()
    for i, (nm, *_rest) in enumerate(feats):
        if geo[i] is None or geo[i][2] != 1:
            continue
        for row in geo[i][3]:
            for m in row:
                if m is None:
                    continue
                if nm == "vanishing-line" and any(Fr(float(v)) != v for v in m):
                    # off the NaN row the homography divides by 632 - v: inexact there, but hundreds of px outside the patch
                    assert max(abs(m[0]), abs(m[1])) > 300, m
                    continue
                for ax_, v in enumerate(m):
                    assert Fr(float(v)) == v and Fr(float(np.float32(float(v)))) == v, (nm, v)  # exact in float64 and float32
                    s = 32 * v
                    if s.denominator == 2:
                        ties["up" if quantise(float(v)) > s else "down"].add((ax_, nm))
                    taps.add((ax_, int(quantise(float(v))) >> 5, bool(int(quantise(float(v))) & 31)))
    for axis in (0, 1):
        assert {a for a, _ in ties["up"]} >= {axis} and {a for a, _ in ties["down"]} >= {axis}
    # taps outside the patch on every side: base index -1 with weight on taps -1 and 0, 40 with weight on 41, and 41 itself
    for axis in (0, 1):
        assert (axis, -1, True) in taps and (axis, 40, True) in taps and (axis, 41, False) in taps and (axis, 39, True) in taps
    nan_rows = [r for r, row in enumerate(g["vanishing-line"][1][3]) if any(m is None for m in row)]
    assert nan_rows == [8]
    # the Q3 zooms: the step of the map is 1/2 for the cartesian feature first in the list, 2 for the one after "zoom-out-2"
    for nm, step in (("q3-cartesian-first-zoom-in", Fr(1, 2)), ("q3-cartesian-after-inverse-depth", Fr(2)), ("zoom-out-4", Fr(4))):
        mp = g[nm][1][3]
        assert mp[0][1][0] - mp[0][0][0] == step, nm
    assert np.count_nonzero(exp) > 0.5 * exp.size


def test_lattice_reference_equals_the_cpp_oracle():
    """The C++ oracle's pred_patch_fc (cv::remap pinned to OpenCV) gives the exact patches bit for bit on every lattice case, and
    np_oracle.pred_patch_maps gives the exact map coordinates bit for bit (NaN on the vanishing line)."""
    from oracle import oracle_py as O

    feats, types, x, p41, vis, h, geo, exp = lattice_case()
    o = O.OracleFilter(CAM_D, quirks=O.Q_ALL, warp_patches=True)
    r, R, uv = init_arrays(feats)
    for i, (t, _) in enumerate(fe[1] for fe in feats):
        o.add_feature(int(t), p41[i], None, r[i], R[i], uv[i])
    o.set_state(x, np.eye(x.size) * 1e-4, prior=True)
    o.search_ic_matches(None)
    fo = o.features()
    assert np.array_equal(fo["has_h"], vis) and np.array_equal(fo["h"][vis], h[vis])
    for i, fe in enumerate(feats):
        if not vis[i]:
            continue
        assert np.array_equal(o.patch_matching(i), exp[i]), fe[0]
        xs, ys, ok, mx, my, _ = NP.pred_patch_maps(CAM_D, x, h[i], NP.xyz_w_for_warp(x, types, i), fe[2], fe[3], fe[4])
        assert (xs, ys, ok) == geo[i][:3] or (ok == geo[i][2] == -1), fe[0]
        if ok == 1:
            for got, a in ((mx, 0), (my, 1)):
                want = np.array([[np.nan if m is None else float(m[a]) for m in row] for row in geo[i][3]])
                if fe[0] == "vanishing-line":  # NaN on the line; the rows beside it divide by 632 - v (inexact)
                    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.allclose(got, want, rtol=1e-12, equal_nan=True)
                else:
                    assert np.array_equal(got, want), fe[0]


# ---- generic geometry on the distorted camera -----------------------------------------------------------------------------------
def rot(axis_angle):
    v = np.asarray(axis_angle, float)
    th = np.linalg.norm(v)
    k = v / th
    Kx = np.array([[0, -k[2], k[1]], [k[2], 0, -k[0]], [-k[1], k[0], 0]])
    return np.eye(3) + math.sin(th) * Kx + (1 - math.cos(th)) * Kx @ Kx


@functools.lru_cache(maxsize=None)
def generic_case(b, N=300):
    """Filter b of the generic batch: a current pose rotated by up to ~15 degrees, N features (every fourth cartesian) spread over
    the image at depths 2..10, each initialised from a pose up to ~25 degrees and ~0.4 away whose camera saw it at uv_init.
    Returns (types, x, p41, feats) with feats = [(name, _, r_init, R_init, uv_init)]."""
    cam = CAM_R
    rng = np.random.default_rng([b, 51])
    Rc = rot(rng.normal(0, 0.15, 3))
    w = math.sqrt(1 + np.trace(Rc)) / 2
    q = np.array([w, (Rc[2, 1] - Rc[1, 2]) / (4 * w), (Rc[0, 2] - Rc[2, 0]) / (4 * w), (Rc[1, 0] - Rc[0, 1]) / (4 * w)])
    rc = rng.normal(0, 0.2, 3)
    types = np.array([1 if i % 4 == 3 else 0 for i in range(N)], np.int32)
    _, _, n = TK.layout(types)
    x = np.zeros(n)
    x[0:3], x[3:7] = rc, q
    feats, off = [], 13
    for i in range(N):
        uv = np.array([rng.uniform(25, COLS - 25), rng.uniform(25, ROWS - 25)])
        p_cam = TK.ray(cam, uv, rng.uniform(2, 10))
        X = rc + Rc @ p_cam
        if types[i] == 1:
            x[off:off + 3] = X
            off += 3
        else:
            a = rc + rng.normal(0, 0.05, 3)
            dvec = X - a
            m = dvec / np.linalg.norm(dvec)
            x[off:off + 3] = a
            x[off + 3] = math.atan2(m[0], m[2])
            x[off + 4] = math.atan2(-m[1], math.hypot(m[0], m[2]))
            x[off + 5] = 1 / np.linalg.norm(dvec)
            off += 6
        Ri = Rc @ rot(rng.normal(0, 0.25, 3))
        ri = rc + rng.normal(0, 0.25, 3)
        pc = Ri.T @ (X - ri)
        uvu = np.array([[cam[4] + pc[0] / pc[2] * cam[6] / cam[7], cam[5] + pc[1] / pc[2] * cam[6] / cam[8]]])
        uvi = NP.distort_fm(cam, uvu)[0] if pc[2] > 0.5 else uv
        feats.append((f"f{i}", None, ri, Ri, uvi))
    p41 = np.stack([np.clip(np.rint(s), 0, 255) for s in synth.smooth_patches(rng, N)]).astype(np.uint8)
    p41[:, 0, 0] = 200
    return types, x, p41, feats


@functools.lru_cache(maxsize=None)
def generic_reference(b):
    """per feature (ok, xs, ys, lo, hi, in_band, vals, window centre) from np_oracle.pred_patch_maps; asserts the 1e-9 margins of
    the gate"""
    types, x, p41, feats = generic_case(b)
    h, vis = NP.predict_h(CAM_R, x, types)
    out = []
    for i, fe in enumerate(feats):
        if not vis[i]:
            out.append(None)
            continue
        for v, lim in ((h[i][0], COLS), (h[i][1], ROWS)):
            assert min(abs(v - HP), abs(v - (lim - HP))) > BAND
        xs, ys, ok, mx, my, c2 = NP.pred_patch_maps(CAM_R, x, h[i], NP.xyz_w_for_warp(x, types, i), fe[2], fe[3], fe[4])
        if ok == 1:
            lo, hi, band, vals = band_values(p41[i], mx, my)
            out.append((ok, xs, ys, lo, hi, band, vals, c2))
        else:
            out.append((ok, xs, ys, None, None, None, None, c2))
    return h, vis, out


def test_generic_cases_stay_off_the_truncation_thresholds():
    """The window ends c2 +- 6 of every generic feature lie more than 1e-9 px from an integer (so truncation is decided), most
    windows are 13 x 13 and most of their pixels sample the patch."""
    for b in range(2):
        types, x, p41, feats = generic_case(b)
        h, vis, ref = generic_reference(b)
        ok = [r for r in ref if r is not None and r[0] == 1]
        assert vis.sum() > 250 and len(ok) > 200
        assert sum(int((r[4] > 0).sum()) for r in ok) > 0.5 * 169 * len(ok)
        for i in np.flatnonzero(vis):
            c2 = ref[i][-1]
            if c2 is not None:
                for v in (c2[0] - HP, c2[0] + HP, c2[1] - HP, c2[1] + HP):
                    assert abs(v - round(v)) > BAND, (b, i)


def test_np_pred_patch_maps_reproduce_the_cpp_oracle():
    """np_oracle.pred_patch_maps followed by the exact remap gives the C++ oracle's patches on the generic maps: bit for bit outside
    the band, one of the two band values inside it, and the same zero patches."""
    from oracle import oracle_py as O

    for b in range(2):
        types, x, p41, feats = generic_case(b)
        h, vis, ref = generic_reference(b)
        o = O.OracleFilter(CAM_R, quirks=O.Q_ALL, warp_patches=True)
        r, R, uv = init_arrays(feats)
        for i in range(len(feats)):
            o.add_feature(int(types[i]), p41[i], None, r[i], R[i], uv[i])
        o.set_state(x, np.eye(x.size) * 1e-4, prior=True)
        o.search_ic_matches(None)
        fo = o.features()
        assert np.array_equal(fo["has_h"], vis)
        TK.assert_close(fo["h"][vis], h[vis], rtol=1e-12, what="h")
        for i in np.flatnonzero(vis):
            check_band(o.patch_matching(i), ref[i], f"filter {b} feature {i}")


def check_band(got, ref, what):
    """got (13 x 13) against one generic reference entry; returns the number of pixels in the band"""
    ok = ref[0]
    got = np.asarray(got, np.float64)
    if ok != 1:
        assert not got.any(), f"{what}: expected the zero patch (ok = {ok})"
        return 0
    _, _, _, lo, hi, band, vals, _ = ref
    hit = (vals == got[None]).any(0)
    assert hit.all(), f"{what}: {int((~hit).sum())} pixels outside the allowed values, first at {np.argwhere(~hit)[0]}"
    assert np.array_equal(got[~band], vals[0][~band]), what
    return int(band.sum())


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lattice_bitwise():
    """Every exact case, bit for bit: sub-pixel offsets, quantisation ties both ways, rotations and a reflection, truncated and
    negative windows, the NaN row on the vanishing line, zooms with taps outside the patch, the Q3 zooms, and the border gate."""
    feats, types, x, p41, vis, h, geo, exp = lattice_case()
    f = capi.Filter(CAM_D, len(feats))
    try:
        run_warp(f, 0, types, x, p41, feats)
        sentinel = np.full((len(feats), 13, 13), -3.0)
        f.upload_patches(sentinel)
        f.set_patch_warp(True)
        f.predict_measurements()
        fg = f.features()
        assert np.array_equal(fg["has_h"], vis) and np.array_equal(fg["h"][vis], h[vis])
        got = f.download_patches()
        exp = exp.copy()
        exp[~vis] = -3.0  # has_h = 0: the uploaded patch survives
        assert_patches_equal(got, exp, [fe[0] for fe in feats], "lattice")
    finally:
        f.close()


def q3_conversion_case():
    """Three features A (inverse depth, X = (0, 0, 3)), B (inverse depth, X = (0, 0, 5), a tiny rho variance: the only linear one)
    and C (cartesian, X = (0, 0, 8)).  After map_inversedepth_to_cartesian converts B, C's XYZ_w is A's point (last_id rewritten
    through map_sync_layout): zoom-out x 2; B (now cartesian) zooms with A's point too.  The prior is uploaded in the converted layout
    before the posterior, so the conversion's last_id is the one the warp reads."""
    old = [("A", id_feat([0.0, 0.0, 3.0]), [0, 0, 1.0], I3, [160.0, 120.0]), ("B", id_feat([0.0, 0.0, 5.0]), [0, 0, 1.0], I3, [160.0, 120.0]),
           ("C", cart_feat([0.0, 0.0, 8.0]), [0, 0, 1.0], I3, [160.0, 120.0])]
    new = [old[0], ("B", cart_feat([0.0, 0.0, 5.0]), [0, 0, 1.0], I3, [160.0, 120.0]), old[2]]
    types_o, x_o = build_filter_state(old)
    types_n, x_n = build_filter_state(new)
    offs, sizes, n = TK.layout(types_o)
    P = np.eye(n) * 1e-4
    P[offs[0] + 5, offs[0] + 5] = 1.0  # A: not linear
    P[offs[1] + 5, offs[1] + 5] = 1e-14  # B: linear
    p41 = patches41(3, 3)
    vis, h, geo, exp = expected_exact(CAM_D, new, types_n, x_n, p41)
    return old, new, types_o, x_o, P, types_n, x_n, p41, vis, exp


def test_q3_conversion_case_zooms():
    old, new, types_o, x_o, P, types_n, x_n, p41, vis, exp = q3_conversion_case()
    assert vis.all()
    for i in range(3):
        _, _, ok, maps = exact_maps(CAM_D, x_n, NP.predict_h(CAM_D, x_n, types_n)[0][i], exact_xyz_w(x_n, types_n, i), new[i][2], I3, new[i][4])
        assert ok == 1 and maps[0][1][0] - maps[0][0][0] == 2  # zoom-out x 2 with A's point; B's own point would give 4/3
    # with the stale last_id (B's point) C's zoom would differ
    _, _, _, maps_b = exact_maps(CAM_D, x_n, (160.0, 120.0), [Fr(0), Fr(0), Fr(5)], new[2][2], I3, new[2][4])
    assert maps_b[0][1][0] - maps_b[0][0][0] != 2


@pytest.mark.gpu
def test_q3_after_inversedepth_to_cartesian():
    old, new, types_o, x_o, P, types_n, x_n, p41, vis, exp = q3_conversion_case()
    f = capi.Filter(CAM_D, 3)
    try:
        f.upload_state(x_n, None, feat_types=types_n, prior=True)
        f.upload_state(x_o, P, feat_types=types_o)
        assert f.map_inversedepth_to_cartesian() == 1
        assert np.array_equal(f.types(), types_n)
        r, R, uv = init_arrays(new)
        f.upload_feature_init(p41, r, R, uv)
        f.set_patch_warp(True)
        f.predict_measurements()
        assert f.features()["has_h"].all()
        assert_patches_equal(f.download_patches(), exp, ["A", "B (converted)", "C"], "after the conversion")
    finally:
        f.close()


BATCHES = {"Nmax7": (7, (7, 5, 7)), "Nmax33": (33, (33, 5, 33))}


@functools.lru_cache(maxsize=None)
def batch_case(key):
    """Per filter of a batch: (feats, types, x, p41, vis, expected).  Identity-lattice features (t = 0: exact) with per-feature
    rotations / reflection and dyadic initial pixels; feature 0 of each filter is never predicted."""
    Nmax, Ns = BATCHES[key]
    out = []
    for b, N in enumerate(Ns):
        rng = np.random.default_rng([Nmax, b, 52])
        feats = [(f"b{b}-0-not-predicted", BEHIND, [0, 0, 0], I3, [100.0, 80.0])]
        for i in range(1, N):
            uvf = [rng.integers(70, 250) + ofs(rng.integers(0, 256)), rng.integers(50, 190) + ofs(rng.integers(0, 256))]
            feats.append((f"b{b}-{i}", id_feat([0.0, 0.0, 2.0]), [0, 0, 0], [I3, ROT90, ROT180, MIRROR][i % 4], uvf))
        types, x = build_filter_state(feats)
        p41 = patches41(100 + b, N)
        vis, h, geo, exp = expected_exact(CAM_D, feats, types, x, p41)
        out.append((feats, types, x, p41, vis, exp))
    return Nmax, Ns, out


@pytest.mark.parametrize("key", list(BATCHES))
def test_batch_cases_cover_every_misalignment(key):
    """On every filter the predicted features' blocks, at (b Nmax + i) 1681 bytes, start at every misalignment 0..3; the last slot
    of the last filter is predicted; the middle filter is shorter than the grid."""
    Nmax, Ns, filt = batch_case(key)
    assert Ns[1] < Nmax and Ns[-1] == Nmax
    for b, (feats, types, x, p41, vis, exp) in enumerate(filt):
        assert not vis[0] and vis[1:].all()
        assert {(b * Nmax + i) % 4 for i in np.flatnonzero(vis)} == {0, 1, 2, 3}
        assert all(exp[i].any() for i in np.flatnonzero(vis))


@pytest.mark.gpu
@pytest.mark.parametrize("key", list(BATCHES))
def test_staging_alignment_and_batch_layout(key):
    """A feature's 41 x 41 block starts (b Nmax + i) 1681 bytes into one allocation: with odd Nmax every misalignment 0..3 occurs on
    every filter, up to the last slot of the last filter.  The middle filter is shorter, so CTAs i >= N run for it and must write
    nothing; a feature that is not predicted keeps its uploaded patch bit for bit."""
    Nmax, Ns, filt = batch_case(key)
    f = capi.Filter(CAM_D, Nmax, batch=len(Ns))
    L = f.L
    try:
        for b, (feats, types, x, p41, vis, exp) in enumerate(filt):
            run_warp(f, b, types, x, p41, feats)
            sentinel = np.full((Nmax, 13, 13), -(b + 1.0))
            assert L.rslam_upload_patches(f.h, b, capi._p(sentinel), Nmax) == 0
        f.set_patch_warp(True)
        f.predict_measurements()
        for b, (feats, types, x, p41, vis, exp) in enumerate(filt):
            N = Ns[b]
            out = np.zeros((Nmax, 13, 13), np.float32)
            assert L.rslam_download_patches(f.h, b, capi._p(out), Nmax) == 0
            assert np.array_equal(f.features(b)["has_h"], vis)
            exp = exp.copy()
            exp[~vis] = -(b + 1.0)  # has_h = 0: the uploaded patch survives
            assert_patches_equal(out[:N], exp, [fe[0] for fe in feats], f"filter {b}")
            assert (out[N:] == -(b + 1.0)).all(), f"filter {b}: slots past N = {N} written"
    finally:
        f.close()


@pytest.mark.gpu
def test_generic_geometry_within_the_band():
    """The distorted camera, rotations of tens of degrees, translations, 300 features per filter in a batch of 2: each pixel equals the
    float64 reference's remap, or one of its two values where a map coordinate lies within 1e-9 px of a quantisation boundary."""
    f = capi.Filter(CAM_R, 300, batch=2)
    try:
        refs = []
        for b in range(2):
            types, x, p41, feats = generic_case(b)
            run_warp(f, b, types, x, p41, feats)
            refs.append(generic_reference(b))
        f.set_patch_warp(True)
        f.predict_measurements()
        in_band = 0
        for b in range(2):
            h, vis, ref = refs[b]
            fg = f.features(b)
            assert np.array_equal(fg["has_h"], vis)
            TK.assert_close(fg["h"][vis], h[vis], what="h")
            got = f.download_patches(b)
            for i in np.flatnonzero(vis):
                in_band += check_band(got[i], ref[i], f"filter {b} feature {i}")
        print(f"generic warp: {in_band} pixels in the 1e-9 px band")
    finally:
        f.close()


@pytest.mark.gpu
def test_search_on_warped_patches():
    """match() on warped patches: the image holds each predicted appearance (rounded to integers) at a candidate of its search region.
    1024 x the warped patch is an integer patch and ZNCC is scale-invariant, so the exact search reference of test_gpu_track_kernels
    applies unchanged: the match must be the exact arg-max wherever that is decided."""
    types, x, p41, feats = generic_case(0)
    N = len(types)
    cam = CAM_R
    rng = np.random.default_rng(53)
    _, _, n = TK.layout(types)
    P = TK.spd(n, TK.map_sd(types, n), rng)
    f = capi.Filter(cam, N)
    try:
        run_warp(f, 0, types, x, p41, feats, prior_P=P)
        f.set_patch_warp(True)
        f.predict_measurements()
        f.set_matches(np.full((N, 2), -7.0), np.zeros(N, bool))  # so that a write by the search shows
        fg = f.features()
        warped = f.download_patches().astype(np.float64)
        img = rng.integers(0, 256, (ROWS, COLS)).astype(np.uint8)
        taken = np.zeros((ROWS, COLS), bool)
        planted = 0
        for k in rng.permutation(N):
            h, S = fg["h"][k], fg["S"][k]
            if not (fg["has_h"][k] and warped[k].std() > 0 and TK.lmax_of(S) < TK.MAX_EIG and HP < h[0] < COLS - HP and HP < h[1] < ROWS - HP):
                continue
            acc = [(j, i) for j, i, ok in TK.gate(h, S, cam)[0] if ok]
            j, i = acc[rng.integers(len(acc))]
            if taken[i - 2 * HP:i + 2 * HP + 1, j - 2 * HP:j + 2 * HP + 1].any():
                continue
            img[i - HP:i + HP + 1, j - HP:j + HP + 1] = np.clip(np.rint(warped[k]), 0, 255).astype(np.uint8)
            taken[i - HP:i + HP + 1, j - HP:j + HP + 1] = True
            planted += 1
        refs, feats_s = [], []
        for k in range(N):
            h, S = fg["h"][k], fg["S"][k]
            p = np.rint(1024 * warped[k]).astype(np.int64)
            assert np.array_equal(p / 1024.0, warped[k])  # warped patches are multiples of 1/1024
            refs.append(TK.search_reference(img, h, S, p, cam) if fg["has_h"][k] else dict(kind="none"))
            feats_s.append((f"f{k}", h, S, p))
        assert planted > 50 and sum(r["kind"] == "one" for r in refs) > 50
        f.set_image(img)
        f.match()
        TK.check_search(f, 0, feats_s, refs, has_h=fg["has_h"])
    finally:
        f.close()
