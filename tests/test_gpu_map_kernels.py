"""The map surgery and feature-initialisation kernels of kernels_map.cuh -- k_map_xform with k_map_prep_convert / k_map_prep_add,
k_map_linearity, k_fast9_score / k_fast9_nms, k_map_box_count and the new feature's record and patch -- against exact and float64
references at the edges where they can go wrong.  Inputs are planted through the C ABI (capi.Filter).

Why the references may be exact.
- Coefficients.  P may be any symmetric matrix, so a probe covariance reads the device's coefficients out exactly: with
  P[ip:ip+6, 0:6] = I the conversion writes P'[ip+r, l] = C[r][l], and with P[0:13, 13:26] = I13 and a zero camera block an addition
  writes P'[n+r, 13+l] = dy/dxv[r][l] and P'[n+r, n+c] = E[max(r,c)][min(r,c)]: every other term of map_comb / map_quad is a product
  with an exact 0 (an exact +-0, with or without FMA contraction).  Values are compared with ==, which takes -0 == +0.
- map_prep_add_dev is written with explicit round-to-nearest products, sums and differences plus IEEE division and sqrt, so a plain
  Python float restatement in the kernel's operation order (`prep_add`) gives the same bits for C, E, x'[0:3], x'[5] and the pose
  record.  Only atan2 (2 ulp in CUDA) is compared with mpmath, at 40 digits, on the very doubles the kernel feeds it.
- map_prep_convert_dev uses CUDA sin / cos (2 ulp each).  Every coefficient is a product of at most two of them, 1 / rho or
  rho * rho and one more rounding, hence within 6 * 2^-52 of the exact value relative (K_CONV), checked against mpmath.
- The linear algebra.  With the coefficients read out, every special entry of P' is sum_k c_k p_k (map_comb) or a quadratic form
  (map_quad) of doubles, whose exact value numpy's long double evaluates to far below the classic rounding bound
  (cnt + 1) u sum |c_k p_k| that the device result must meet.  Copied entries are copies, bit for bit, and P' is bitwise symmetric.
- The linearity index is planted at 0.1 (1 +- 1e-9) in mpmath, a margin five orders of magnitude above its float64 error (checked on
  the CPU), so which feature k_map_linearity picks is exact.
- FAST-9 is integer arithmetic: oracle_py.fast9, pinned to cv2 with order included, is the exact reference.  The designed tiles
  reach the score edges according to a plain numpy scorer (`fast_scores`), which a CPU test checks.
- The sampling box uses a dyadic pinhole camera (k1 = k2 = 0, f / dx = 256) and the identity pose, where the predicted pixel of a
  cartesian feature is exact, so features sit exactly on, or 2^-20 px inside or outside, each edge of the box.  The +-60 degree gates
  are planted 1e-9 rad off in mpmath."""
import math

import numpy as np
import pytest

from oracle import np_oracle as NP
from oracle import oracle_py as O
from ransac_slam_b200 import synth

U = 2.0**-53
K_CONV = 6
CAM_R = synth.Camera().as9()
CAM_A = CAM_R.copy()
CAM_A[4:6] = [151.3, 117.9]  # another principal point (dx == dy: the reference's K takes f / dx for both rows, src/System.cpp:58)
CAM_D = np.array([0.0, 0.0, 1024, 1024, 512.0, 512.0, 1.0, 2.0**-8, 2.0**-8])  # dyadic pinhole, f / dx = 256
CAM_W = np.array([0.0, 0.0, 1024, 1024, 512.0, 512.0, 1.0, 2.0**-10, 2.0**-10])  # f / dx = 1024: the image edges lie inside +-60 deg


def _filter(cam9, max_features, std_z=1.0, batch=1):
    from ransac_slam_b200 import capi

    return capi.Filter(cam9, max_features, batch=batch, std_z=std_z)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _layout(types):
    offs, off = [], 13
    for t in types:
        offs.append(off)
        off += 6 if t == 0 else 3
    return offs, off


def _exact_eq(a, b):
    """== entry by entry (-0 == +0) and the same NaN pattern"""
    a, b = np.asarray(a, float), np.asarray(b, float)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


# ---- restatements: one body per kernel, run in float64 (the kernel's operation order) or in mpmath at 40 digits -------------------
class F64:
    mul = staticmethod(lambda a, b: a * b)
    add = staticmethod(lambda a, b: a + b)
    sub = staticmethod(lambda a, b: a - b)
    div = staticmethod(lambda a, b: a / b)
    sqrt = staticmethod(math.sqrt)
    sin = staticmethod(math.sin)
    cos = staticmethod(math.cos)
    atan2 = staticmethod(math.atan2)
    num = staticmethod(float)


class MP:
    import mpmath as _m

    ctx = _m.mp.clone()
    ctx.dps = 40
    mul = staticmethod(lambda a, b: MP.ctx.fmul(a, b))
    add = staticmethod(lambda a, b: MP.ctx.fadd(a, b))
    sub = staticmethod(lambda a, b: MP.ctx.fsub(a, b))
    div = staticmethod(lambda a, b: MP.ctx.fdiv(a, b))
    sqrt = staticmethod(lambda a: MP.ctx.sqrt(a))
    sin = staticmethod(lambda a: MP.ctx.sin(a))
    cos = staticmethod(lambda a: MP.ctx.cos(a))
    atan2 = staticmethod(lambda a, b: MP.ctx.atan2(a, b))
    num = staticmethod(lambda a: MP.ctx.mpf(float(a)))


def lin_index(A, xc, y, var_rho):
    """map_is_linear_dev's linearity index (src/Map.cpp:113-148)"""
    xc, y = [A.num(v) for v in xc], [A.num(v) for v in y]
    std_d = A.div(A.sqrt(A.num(var_rho)), A.mul(y[5], y[5]))
    mi = [A.mul(A.cos(y[4]), A.sin(y[3])), -A.sin(y[4]), A.mul(A.cos(y[4]), A.cos(y[3]))]
    a = n1 = n2 = A.num(0.0)
    for k in range(3):
        xo = A.add(y[k], A.div(mi[k], y[5]))
        d1, d2 = A.sub(xo, y[k]), A.sub(xo, xc[k])
        a, n1, n2 = A.add(a, A.mul(d1, d2)), A.add(n1, A.mul(d1, d1)), A.add(n2, A.mul(d2, d2))
    cos_alpha = A.div(a, A.mul(A.sqrt(n1), A.sqrt(n2)))
    return A.div(A.mul(A.mul(A.num(4.0), std_d), cos_alpha), A.sqrt(n2))


def prep_convert(A, y):
    """map_prep_convert_dev: C[3][6] of the conversion (src/Map.cpp:150-169) and the cartesian point xs[3]"""
    th, ph, rho = (A.num(v) for v in y[3:6])
    mi = [A.mul(A.cos(ph), A.sin(th)), -A.sin(ph), A.mul(A.cos(ph), A.cos(th))]
    dmt = [A.mul(A.cos(ph), A.cos(th)), A.num(0.0), -A.mul(A.cos(ph), A.sin(th))]
    dmp = [-A.mul(A.sin(ph), A.sin(th)), -A.cos(ph), -A.mul(A.sin(ph), A.cos(th))]
    one = A.num(1.0)
    C = [[one if r == c else A.num(0.0) for c in range(3)] + [A.mul(A.div(one, rho), dmt[r]), A.mul(A.div(one, rho), dmp[r]),
                                                           A.div(-mi[r], A.mul(rho, rho))] for r in range(3)]
    xs = [A.add(A.num(y[r]), A.div(mi[r], rho)) for r in range(3)]
    return C, xs


def prep_add(A, Xv, cam9, ud, vd, std_pxl, std_rho=1.0, initial_rho=1.0, dgc_fill="reference"):
    """map_prep_add_dev: hinv (src/ExtendKF.cpp:236-265) and the Jacobians of add_a_feature_covariance_inverse_depth
    (src/Map.cpp:339-386), operation for operation.  Returns dict(C = dy/dxv [6][13], E [6][6], xs [6], pose14 [14], dy_dhd [6][3],
    atan2 = the two (y, x) argument pairs)."""
    m, a, s, d = A.mul, A.add, A.sub, A.div
    k1, k2, _, _, Cx, Cy, f, dx, dy = (A.num(v) for v in cam9)
    one, two, zero = A.num(1.0), A.num(2.0), A.num(0.0)
    fku, fkv = m(f, d(one, dx)), m(f, d(one, dy))  # CamDev, as rslam_create fills it
    ud, vd = A.num(ud), A.num(vd)
    qr, qx, qy, qz = (A.num(v) for v in Xv[3:7])
    R = [s(s(a(m(qr, qr), m(qx, qx)), m(qy, qy)), m(qz, qz)), m(two, s(m(qx, qy), m(qr, qz))), m(two, a(m(qz, qx), m(qr, qy))),
         m(two, a(m(qx, qy), m(qr, qz))), s(a(s(m(qr, qr), m(qx, qx)), m(qy, qy)), m(qz, qz)), m(two, s(m(qy, qz), m(qr, qx))),
         m(two, s(m(qz, qx), m(qr, qy))), m(two, a(m(qy, qz), m(qr, qx))), a(s(s(m(qr, qr), m(qx, qx)), m(qy, qy)), m(qz, qz))]
    xd, yd = m(s(ud, Cx), dx), m(s(vd, Cy), dy)
    rd = A.sqrt(a(m(xd, xd), m(yd, yd)))
    D = a(a(one, m(m(k1, rd), rd)), m(m(m(m(k2, rd), rd), rd), rd))
    uu, vu = a(d(m(xd, D), dx), Cx), a(d(m(yd, D), dy), Cy)
    gc = [d(-s(Cx, uu), fku), d(-s(Cy, vu), fkv), one]
    gw = [a(a(m(R[3 * k], gc[0]), m(R[3 * k + 1], gc[1])), m(R[3 * k + 2], gc[2])) for k in range(3)]
    Xw, Yw, Zw = gw
    xz2 = a(m(Xw, Xw), m(Zw, Zw))
    n2, sxz = a(xz2, m(Yw, Yw)), A.sqrt(xz2)
    xs = [A.num(Xv[0]), A.num(Xv[1]), A.num(Xv[2]), A.atan2(Xw, Zw), A.atan2(-Yw, sxz), A.num(initial_rho)]
    g = gc
    dq = [None] * 12
    dq[0] = m(two, a(s(m(qr, g[0]), m(qz, g[1])), m(qy, g[2])))
    dq[4] = m(two, s(a(m(qz, g[0]), m(qr, g[1])), m(qx, g[2])))
    dq[8] = m(two, a(a(m(-qy, g[0]), m(qx, g[1])), m(qr, g[2])))
    dq[1] = m(two, a(a(m(qx, g[0]), m(qy, g[1])), m(qz, g[2])))
    dq[5] = m(two, s(s(m(qy, g[0]), m(qx, g[1])), m(qr, g[2])))
    dq[9] = m(two, s(a(m(qz, g[0]), m(qr, g[1])), m(qx, g[2])))
    dq[2] = m(two, a(a(m(-qy, g[0]), m(qx, g[1])), m(qr, g[2])))
    dq[6] = m(two, a(a(m(qx, g[0]), m(qy, g[1])), m(qz, g[2])))
    dq[10] = m(two, s(a(m(-qr, g[0]), m(qz, g[1])), m(qy, g[2])))
    dq[3] = m(two, a(s(m(-qz, g[0]), m(qr, g[1])), m(qx, g[2])))
    dq[7] = m(two, a(s(m(qr, g[0]), m(qz, g[1])), m(qy, g[2])))
    dq[11] = m(two, a(a(m(qx, g[0]), m(qy, g[1])), m(qz, g[2])))
    dth = [d(Zw, xz2), zero, d(-Xw, xz2)]
    dph = [d(m(Xw, Yw), m(n2, sxz)), d(-sxz, n2), d(m(Zw, Yw), m(n2, sxz))]
    C = [[zero] * 13 for _ in range(6)]
    for r in range(3):
        C[r][r] = one
    for c in range(4):
        C[3][3 + c] = a(a(m(dth[0], dq[c]), m(dth[1], dq[4 + c])), m(dth[2], dq[8 + c]))
        C[4][3 + c] = a(a(m(dph[0], dq[c]), m(dph[1], dq[4 + c])), m(dph[2], dq[8 + c]))
    ja, jb = s(ud, Cx), s(vd, Cy)
    adx, bdy = m(ja, dx), m(jb, dy)
    rd2 = a(m(adx, adx), m(bdy, bdy))
    gg = a(k1, m(m(two, k2), rd2))
    cc = a(a(one, m(k1, rd2)), m(m(k2, rd2), rd2))
    J = [a(cc, m(m(ja, gg), m(m(m(two, ja), dx), dx))), m(m(ja, gg), m(m(m(two, jb), dy), dy)),
         m(m(jb, gg), m(m(m(two, ja), dx), dx)), a(cc, m(m(jb, gg), m(m(m(two, jb), dy), dy)))]
    tR = [[a(a(m(dt[0], R[c]), m(dt[1], R[3 + c])), m(dt[2], R[6 + c])) for c in range(3)] for dt in (dth, dph)]
    # quirk Q16: Eigen fills the comma-initialised 3 x 2 dgc_dhu row by row, [1/fku 0; 0 0; 1/fkv 0] (src/Map.cpp:375-379)
    assert dgc_fill == "reference"
    tg = [[a(m(tR[r][0], d(one, fku)), m(tR[r][2], d(one, fkv))), zero] for r in range(2)]
    dy_dhd = [[zero] * 3 for _ in range(6)]
    for r in range(2):
        for c in range(2):
            dy_dhd[3 + r][c] = a(m(tg[r][0], J[c]), m(tg[r][1], J[2 + c]))
    dy_dhd[5][2] = one
    pad = [m(A.num(std_pxl), A.num(std_pxl)), m(A.num(std_pxl), A.num(std_pxl)), m(A.num(std_rho), A.num(std_rho))]
    E = [[zero] * 6 for _ in range(6)]
    for r in range(6):
        for c in range(6):
            acc = zero
            for k in range(3):
                acc = a(acc, m(m(dy_dhd[r][k], pad[k]), dy_dhd[c][k]))
            E[r][c] = acc
    pose14 = [A.num(Xv[0]), A.num(Xv[1]), A.num(Xv[2])] + R + [ud, vd]
    return dict(C=C, E=E, xs=xs, pose14=pose14, dy_dhd=dy_dhd, atan2=((Xw, Zw), (-Yw, sxz)))


def _arr(v):
    return np.array(v, dtype=float)


def _ulps(got, exact):
    """|got - exact| in units of the last place of float(exact)"""
    return float(abs(MP.ctx.mpf(float(got)) - exact) / math.ulp(float(exact))) if float(exact) != 0 else (0.0 if got == 0 else math.inf)


# ---- cases ----------------------------------------------------------------------------------------------------------------------
def _q(*v):
    v = np.array(v, float)
    return v / np.linalg.norm(v)


def _camera_x(q, r=(0.1, -0.2, 0.3)):
    x = np.zeros(13)
    x[0:3] = r
    x[3:7] = q
    x[7:13] = [0.01, -0.02, 0.005, 0.001, -0.002, 0.003]
    return x


def add_cases():
    """(name, cam9, camera state, (ud, vd), std_z) for the addition: principal point, the four corners, both sides of the atan2
    branch cut (Zw < 0), the pole (xz2 ~ 1e-10 n2), qr < 0 and std_z != 1"""
    rng = np.random.default_rng(3)
    q0 = _q(0.97, 0.05, -0.2, 0.1)
    back = _q(1e-3, 0.0, 1.0, 0.0)  # about 180 degrees around y: the ray points along -Z
    pole = _q(1.0, 1.0, 0.0, 0.0)  # 90 degrees around x: a ray near the optical axis maps onto -Y
    cases = []
    for cam, tag in ((CAM_A, "dxdy"), (CAM_R, "real")):
        Cx, Cy, cols, rows = cam[4], cam[5], int(cam[3]), int(cam[2])
        cases += [(f"{tag}-principal", cam, _camera_x(q0), (Cx, Cy), 1.0)]
        cases += [(f"{tag}-corner{k}", cam, _camera_x(q0), uv, 1.0) for k, uv in enumerate([(0.0, 0.0), (cols - 1.0, 0.0), (0.0, rows - 1.0), (cols - 1.0, rows - 1.0)])]
    cases += [("cut+", CAM_A, _camera_x(back), (CAM_A[4] + 1.0, 77.0), 1.0), ("cut-", CAM_A, _camera_x(back), (CAM_A[4] - 1.0, 77.0), 1.0)]
    cases += [("pole", CAM_A, _camera_x(pole), (CAM_A[4] + 0.002, CAM_A[5] + 0.002), 1.0)]
    cases += [("qr<0", CAM_A, _camera_x(-q0), (201.0, 77.0), 1.0), ("std_z", CAM_A, _camera_x(q0), (64.5, 150.25), 1.7)]
    cases += [(f"random{k}", CAM_A, _camera_x(_q(*rng.normal(0, 1, 4)), rng.normal(0, 1, 3)), tuple(rng.uniform(0, 320, 2)), float(rng.uniform(0.5, 2))) for k in range(3)]
    return cases


def _probe_add_state(Xv, N=3, rng=None):
    """camera Xv, N inverse-depth features, P[0:13, 13:26] = I13 (and its transpose), a zero camera block, 1 elsewhere on the diagonal"""
    rng = rng or np.random.default_rng(0)
    n = 13 + 6 * N
    x = np.r_[Xv, np.concatenate([np.r_[rng.normal(0, 1, 3), rng.uniform(-1, 1, 2), rng.uniform(0.1, 1)] for _ in range(N)])]
    P = np.eye(n)
    P[0:13, 0:13] = 0
    P[0:13, 13:26] = np.eye(13)
    P[13:26, 0:13] = np.eye(13)
    return x, np.asfortranarray(P)


def _read_add(x, P, Pn, xn):
    n = x.size
    return Pn[n:n + 6, 13:26], Pn[n:n + 6, n:n + 6], xn[n:n + 6]


def _probe_convert_state(Xc, y, extra=1):
    """camera Xc, feature 0 = y (then `extra` features with a huge rho variance), P[ip:ip+6, 0:6] = I and a small P[ip+5, ip+5]"""
    N = 1 + extra
    n = 13 + 6 * N
    x = np.r_[Xc, y, np.tile([0.0, 0.0, 0.0, 0.1, 0.1, 0.5], extra)]
    P = np.eye(n) * 1e6
    P[0:13, 0:13] = np.eye(13)
    P[13:19, 0:6] = np.eye(6)
    P[0:6, 13:19] = np.eye(6)
    P[18, 18] = 1e-12
    return x, np.asfortranarray(P)


def conv_cases():
    rng = np.random.default_rng(5)
    ys = [np.r_[rng.normal(0, 1, 3), rng.uniform(-3, 3), rng.uniform(-1.5, 1.5), rng.uniform(0.05, 2)] for _ in range(6)]
    ys += [np.r_[0.1, 0.2, 0.3, 0.0, 0.0, 1.0], np.r_[0.0, 0.0, 0.0, np.pi / 2, -np.pi / 2 + 1e-3, 0.3], np.r_[1.0, -1.0, 2.0, -2.9, 1.2, -0.4]]
    return ys


# ---- CPU self-checks of the restatements ----------------------------------------------------------------------------------------
def _rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def test_restatements_match_the_oracle():
    """prep_add / prep_convert in float64 against the C++ oracle (same probe read-out), and against their own mpmath runs"""
    for name, cam, Xv, uv, std_z in add_cases():
        x, P = _probe_add_state(Xv)
        o = O.OracleFilter(cam, std_z=std_z)
        for i in range(3):
            o.add_feature(0)
        o.set_state(x, P)
        assert o.map_add_feature(np.array(uv)) == 3
        xo, Po = o.get_state()
        Co, Eo, xso = _read_add(x, P, Po, xo)
        r = prep_add(F64, Xv, cam, uv[0], uv[1], std_z)
        assert _rel(r["C"], Co) < 1e-13 and _rel(r["E"], Eo) < 1e-13 and _rel(r["xs"], xso) < 1e-13, name
        _, pose = o.feature_init(3)
        assert _rel(r["pose14"], pose) < 1e-13, name
        if name != "pole":  # near the pole, gw's cancellation (1e-16 against 1e-5) makes float64 itself relatively inaccurate
            rm = prep_add(MP, Xv, cam, uv[0], uv[1], std_z)
            for k in ("C", "E", "xs"):
                assert _rel(r[k], [[float(v) for v in row] for row in rm[k]] if k != "xs" else [float(v) for v in rm[k]]) < 1e-12, (name, k)
        # and the independent numpy restatement of the same Jacobians (quirk Q16 fill)
        c = synth.Camera(*[cam[0], cam[1], int(cam[2]), int(cam[3])] + list(cam[4:]))
        dxv, dhd = synth.feature_init_jacobians(c, np.array(uv), Xv, reference_fill=True)
        assert _rel(r["C"], dxv) < 1e-11 and _rel(r["dy_dhd"], dhd) < 1e-11, name
    Xc = _camera_x(_q(0.9, 0.1, 0.3, -0.2))
    for y in conv_cases():
        x, P = _probe_convert_state(Xc, y)
        o = O.OracleFilter(CAM_R)
        for i in range(2):
            o.add_feature(0)
        o.set_state(x, P)
        assert o.map_inversedepth_to_cartesian() == 0
        xo, Po = o.get_state()
        C, xs = prep_convert(F64, y)
        assert _rel(C, Po[13:16, 0:6]) < 1e-13 and _rel(xs, xo[13:16]) < 1e-13
        Cm, xm = prep_convert(MP, y)
        assert _rel(C, [[float(v) for v in row] for row in Cm]) < 1e-14 and _rel(xs, [float(v) for v in xm]) < 1e-14


# ---- 2. coefficients on the device --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_add_coefficients_bitwise():
    """C (dy/dxv), E, x'[0:3], x'[5] and pose14 bit for bit against the float64 restatement; the two angles within 2 ulp of atan2"""
    worst = 0.0
    for name, cam, Xv, uv, std_z in add_cases():
        x, P = _probe_add_state(Xv)
        g = _filter(cam, 4, std_z=std_z)
        g.upload_state(x, P)
        assert g.map_add_feature(np.array(uv)) == 3
        xn, Pn = g.download_state()
        C, E, xs = _read_add(x, P, Pn, xn)
        r = prep_add(F64, Xv, cam, uv[0], uv[1], std_z)
        Er = _arr(r["E"])
        assert _exact_eq(C, r["C"]), (name, C, _arr(r["C"]))
        assert _exact_eq(E, np.tril(Er) + np.tril(Er, -1).T), name  # the lower triangle, mirrored
        assert _exact_eq(xs[[0, 1, 2, 5]], _arr(r["xs"])[[0, 1, 2, 5]]), name
        for k, (yy, xx) in zip((3, 4), r["atan2"]):
            e = MP.ctx.atan2(MP.ctx.mpf(yy), MP.ctx.mpf(xx))
            worst = max(worst, _ulps(xs[k], e))
            assert _ulps(xs[k], e) <= 2, (name, k, xs[k], e)
        _, pose = g.feature_init(3)
        assert _exact_eq(pose, r["pose14"]), name
        assert np.array_equal(_bits(Pn), _bits(Pn.T)), name
        g.close()


@pytest.mark.gpu
def test_convert_coefficients_within_bound():
    """C and x' of the conversion within K_CONV * 2^-52 (relative) of mpmath; the identity block exact"""
    Xc = _camera_x(_q(0.9, 0.1, 0.3, -0.2))
    for y in conv_cases():
        x, P = _probe_convert_state(Xc, y)
        g = _filter(CAM_R, 2)
        g.upload_state(x, P)
        assert g.map_inversedepth_to_cartesian() == 0
        xn, Pn = g.download_state()
        C, xs = Pn[13:16, 0:6], xn[13:16]
        Cm, xm = prep_convert(MP, y)
        for r in range(3):
            for c in range(6):
                e = Cm[r][c]
                assert abs(MP.ctx.mpf(float(C[r, c])) - e) <= K_CONV * 2.0**-52 * abs(e), (y, r, c, C[r, c], e)
            mr = abs(MP.ctx.mpf(float(xs[r])) - y[r])  # |mi / rho|, near enough for the bound
            assert abs(MP.ctx.mpf(float(xs[r])) - xm[r]) <= K_CONV * 2.0**-52 * mr + 2.0**-52 * abs(xm[r]), (y, r)
        assert _exact_eq(C[:, 0:3], np.eye(3))
        assert np.array_equal(_bits(Pn), _bits(Pn.T))
        g.close()


# ---- 1. the T P T^T pass against an exact reference ---------------------------------------------------------------------------------
def _probe_C_convert(x, types, i):
    """the device's conversion coefficients for feature i of state x: the same y as feature 0 of a small probe map"""
    offs, _ = _layout(types)
    y = x[offs[i]:offs[i] + 6]
    xp, Pp = _probe_convert_state(x[:13], y)
    g = _filter(CAM_R, 2)
    g.upload_state(xp, Pp)
    assert g.map_inversedepth_to_cartesian() == 0
    xn, Pn = g.download_state()
    g.close()
    return Pn[13:16, 0:6].copy(), xn[13:16].copy()


def _check_special(Pold, Pnew, sp_new, src_old, C, copy_new, copy_old, E=None):
    """special rows sp_new of Pnew against the exact sum_k C[r][k] Pold[src_old[k], .] within (cnt + 1) u sum |c_k p_k|; the
    special x special block against C Pss C^T + E within (2 cnt + 2) u (|C| |Pss| |C|^T + |E|)"""
    assert np.finfo(np.longdouble).nmant >= 63
    cnt = len(src_old)
    Cl = np.asarray(C, np.longdouble)
    Pl = np.asarray(Pold, np.longdouble)
    blk = Pl[np.ix_(src_old, copy_old)]
    exact = Cl @ blk
    bound = (cnt + 1) * U * (np.abs(Cl) @ np.abs(blk)) * (1 + 2.0**-10)
    got = Pnew[np.ix_(sp_new, copy_new)]
    err = np.abs(got.astype(np.longdouble) - exact)
    assert np.all(err <= bound), float(np.max(err / np.maximum(bound, 1e-300)))
    Pss = Pl[np.ix_(src_old, src_old)]
    El = np.zeros((len(sp_new),) * 2, np.longdouble) if E is None else np.asarray(E, np.longdouble)
    exact = Cl @ Pss @ Cl.T + El
    bound = (2 * cnt + 2) * U * (np.abs(Cl) @ np.abs(Pss) @ np.abs(Cl).T + np.abs(El)) * (1 + 2.0**-10)
    err = np.abs(Pnew[np.ix_(sp_new, sp_new)].astype(np.longdouble) - exact)
    assert np.all(err <= bound)


def _check_op(op, x, P, types, xn, Pn, arg):
    """x', P' after `op` against the exact reference: copies bitwise, special entries within the bound, P' bitwise symmetric"""
    n = x.size
    offs, _ = _layout(types)
    assert np.array_equal(_bits(Pn), _bits(Pn.T)), op
    if op == "delete":
        i = arg
        sz = 6 if types[i] == 0 else 3
        keep = np.r_[0:offs[i], offs[i] + sz:n]
        assert np.array_equal(_bits(Pn), _bits(P[np.ix_(keep, keep)])) and np.array_equal(_bits(xn), _bits(x[keep])), op
        return
    if op == "convert":
        i, C, xs = arg
        ip = offs[i]
        copy_new = np.r_[0:ip, ip + 3:n - 3]
        copy_old = np.r_[0:ip, ip + 6:n]
        sp_new, src, E = np.arange(ip, ip + 3), np.arange(ip, ip + 6), None
    else:
        C, E, xs = arg
        copy_new = copy_old = np.arange(n)
        sp_new, src = np.arange(n, n + 6), np.arange(13)
    assert np.array_equal(_bits(Pn[np.ix_(copy_new, copy_new)]), _bits(P[np.ix_(copy_old, copy_old)])), op
    assert np.array_equal(_bits(xn[copy_new]), _bits(x[copy_old])), op
    if op == "add":  # xs from the float64 restatement: the two angles come from atan2 (CUDA 2 ulp, libm 1 ulp)
        assert _exact_eq(xn[sp_new][[0, 1, 2, 5]], xs[[0, 1, 2, 5]]), op
        assert all(abs(a - b) <= 3 * math.ulp(b) for a, b in zip(xn[sp_new][3:5], xs[3:5])), (op, xn[sp_new], xs)
    else:
        assert _exact_eq(xn[sp_new], xs), op
    _check_special(P, Pn, sp_new, src, C, copy_new, copy_old, E)


def _spd_state(N, seed, cartesian=(), convert=None):
    """random SPD state of N features; `cartesian` keep 3 of their 6 rows; feature `convert` gets a rho variance that passes the
    linearity test"""
    scene, x, P = synth.random_spd_state(N, seed=seed)
    types = np.zeros(N, np.int32)
    keep = np.ones(x.size, bool)
    for i in cartesian:
        types[i] = 1
        keep[13 + 6 * i + 3:13 + 6 * i + 6] = False
    if convert is not None:
        ip = 13 + 6 * convert
        s = 1e-3 / np.sqrt(P[ip + 5, ip + 5])
        P[ip + 5, :] *= s
        P[:, ip + 5] *= s
    return x[keep], np.asfortranarray(P[np.ix_(keep, keep)]), types


def _first_linear(x, P, types):
    offs, _ = _layout(types)
    for i, t in enumerate(types):
        if t == 0 and lin_index(F64, x[:3], x[offs[i]:offs[i] + 6], P[offs[i] + 5, offs[i] + 5]) < 0.1:
            return i
    return -1


class _Map:
    """a per-filter handle and the host copy of the state it holds"""

    def __init__(self, x, P, types, max_features, std_z=1.0):
        self.g = _filter(CAM_R, max_features, std_z=std_z)
        self.g.upload_state(x, P, feat_types=types)
        self.x, self.P, self.types = x, P, list(types)

    def op(self, op, arg=None):
        g = self.g
        if op == "delete":
            g.map_delete_feature(arg)
            a = arg
        elif op == "convert":
            i = _first_linear(self.x, self.P, self.types)
            assert i == arg
            C, xs = _probe_C_convert(self.x, self.types, i)
            assert g.map_inversedepth_to_cartesian() == i
            a = (i, C, xs)
        else:
            r = prep_add(F64, self.x[:13], CAM_R, arg[0], arg[1], g.par.std_z)
            assert g.map_add_feature(np.array(arg)) == len(self.types)
            a = (_arr(r["C"]), _arr(r["E"]), _arr(r["xs"]))
        xn, Pn = g.download_state()
        _check_op(op, self.x, self.P, self.types, xn, Pn, a)
        if op == "delete":
            del self.types[arg]
        elif op == "convert":
            self.types[arg] = 1
        else:
            self.types.append(0)
        assert list(g.types()) == self.types
        self.x, self.P = xn, Pn


@pytest.mark.gpu
def test_surgery_chain_exact_and_symmetric():
    """conversion of feature 0, of the last feature behind cartesian ones, deletion of an inverse-depth block and of a cartesian
    block at the end, additions; P' checked after every step, and the chain ends in a checkpoint, which needs P bitwise symmetric"""
    x, P, types = _spd_state(12, 31, cartesian=(3, 7, 11), convert=0)
    m = _Map(x, P, types, 16, std_z=1.3)
    m.op("convert", 0)
    m.op("delete", 5)
    m.op("add", (201.0, 77.0))
    # the new (last) feature passes the linearity test once its rho variance is small: make it so and convert it
    offs, n = _layout(m.types)
    ip = offs[-1]
    s = 1e-3 / math.sqrt(m.P[ip + 5, ip + 5])
    P2 = m.P.copy()
    P2[ip + 5, :] *= s
    P2[:, ip + 5] *= s
    P2[ip + 5, ip + 5] = m.P[ip + 5, ip + 5] * s * s
    m.g.upload_state(m.x, P2, feat_types=m.types)
    m.P = P2
    m.op("convert", len(m.types) - 1)
    m.op("delete", len(m.types) - 1)  # a 3-wide cartesian block at the end
    m.op("add", (0.0, 239.0))
    buf = m.g.save()
    from ransac_slam_b200 import capi

    hdr, fl = capi.read_checkpoint(buf)
    assert np.array_equal(_bits(fl[0]["P"]), _bits(m.P))


@pytest.mark.gpu
def test_delete_to_camera_then_add_to_empty_map():
    x, P, types = _spd_state(4, 33, cartesian=(1, 3))
    m = _Map(x, P, types, 4)
    for i in (3, 0, 1, 0):
        m.op("delete", i)
    assert m.x.size == 13 and m.g.N == 0
    m.op("add", (CAM_R[4], CAM_R[5]))
    m.op("add", (319.0, 0.0))


def _types_for(n):
    """N features (at most one cartesian, last) with 13 + sum(sizes) == n"""
    b = ((n - 13) // 3) % 2
    a = (n - 13 - 3 * b) // 6
    return a + b, tuple(range(a, a + b))


@pytest.mark.gpu
@pytest.mark.parametrize("n_new", [253, 256, 259])  # n = 13 + 6 a + 3 b is 1 mod 3, and so is every n'
@pytest.mark.parametrize("op", ["add", "convert", "delete"])
def test_cta_boundary(op, n_new):
    n = {"add": n_new - 6, "convert": n_new + 3, "delete": n_new + 6}[op]
    N, cart = _types_for(n)
    last_idd = N - 1 - len(cart)  # the converted / deleted feature: the last inverse-depth one, before a cartesian tail
    x, P, types = _spd_state(N, 40 + n_new, cartesian=cart, convert=last_idd if op == "convert" else None)
    assert x.size == n
    m = _Map(x, P, types, N + 1)
    m.op(op, {"add": (100.5, 200.25), "convert": last_idd, "delete": last_idd}[op])
    assert m.x.size == n_new


@pytest.mark.gpu
def test_large_map_conversion():
    """N = 2000 (P = 1.15 GB, assembled on the device): the three special rows within the bound, everything else bitwise"""
    import torch

    N = 2000
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
    dev = torch.device("cuda", 0)
    P0 = synth.assemble_P_torch(scene, dev)
    n = scene.x0.size
    i = 1500
    ip = 13 + 6 * i
    s = 1e-3 / torch.sqrt(P0[ip + 5, ip + 5])
    P0[ip + 5, :] *= s
    P0[:, ip + 5] *= s
    x0 = scene.x0
    diag = torch.diagonal(P0).cpu().numpy()
    types = [0] * N
    assert min(k for k in range(N) if lin_index(F64, x0[:3], x0[13 + 6 * k:19 + 6 * k], diag[18 + 6 * k]) < 0.1) == i
    C, xs = _probe_C_convert(x0, types, i)
    g = _filter(cam.as9(), N)
    xd = torch.from_numpy(x0).to(dev)
    g.upload_state_device(xd.data_ptr(), P0.data_ptr(), n, n, N)
    assert g.map_inversedepth_to_cartesian() == i
    xn, Pn = g.download_state()
    g.close()
    Ph = P0.cpu().numpy()
    del P0
    _check_op("convert", x0, Ph, types, xn, Pn, (i, C, xs))


# ---- 3. which feature is converted ------------------------------------------------------------------------------------------------
def plant_var(xc, y, target):
    """the rho variance that puts the linearity index at `target` (mpmath; the index is proportional to sqrt(var))"""
    k = lin_index(MP, xc, y, 1.0)
    assert k * target > 0
    return float((MP.ctx.mpf(target) / k) ** 2)


LO, HI = 0.1 * (1 - 1e-9), 0.1 * (1 + 1e-9)


def linearity_case(name):
    """(x, P, types, expected index) of each case; every inverse-depth feature planted at LO (qualifies) or HI (does not)"""
    rng = np.random.default_rng(LIN_CASES.index(name))
    N = {"127+128": 200, "128+300": 320, "cartesian": 40, "negative-rho": 12, "none": 150}[name]
    qual = {"127+128": (127, 128), "128+300": (128, 300), "cartesian": (30,), "negative-rho": (7,), "none": ()}[name]
    cart = {"cartesian": (4, 20)}.get(name, ())
    types = np.array([1 if i in cart else 0 for i in range(N)], np.int32)
    offs, n = _layout(types)
    x = np.zeros(n)
    x[0:3] = [0.05, -0.1, 0.2]
    x[3:7] = _q(0.99, 0.02, 0.1, 0.0)
    P = np.eye(n) * 1e-4
    for i in range(N):
        o = offs[i]
        if types[i] == 1:
            x[o:o + 3] = rng.normal(0, 1, 3)
            continue
        rho = rng.uniform(0.2, 2.0) * (-1 if name == "negative-rho" and i % 2 else 1)
        x[o:o + 6] = np.r_[x[0:3] + rng.normal(0, 0.01, 3), rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.4), rho]
    for i in cart:
        # the six numbers a misread cartesian slot would give (its point, then the next feature's first three rows) qualify by far
        o = offs[i]
        x[o + 3:o + 6] = [0.1, 0.05, 0.5]  # the next feature's anchor point: a valid position, and (theta, phi, rho) that qualify
        P[o + 5, o + 5] = 1e-14
    for i in range(N):
        o = offs[i]
        if types[i] == 0:
            P[o + 5, o + 5] = plant_var(x[:3], x[o:o + 6], LO if i in qual else HI)
    exp = min(qual) if qual else -1
    return x, np.asfortranarray(P), types, exp


LIN_CASES = ["127+128", "128+300", "cartesian", "negative-rho", "none"]


def test_linearity_planting_margins():
    """the planted indices sit 1e-9 (relative) off 0.1 in mpmath, far beyond the float64 restatement's error; the float64 choice is
    the expected one, and a cartesian slot read as inverse depth would qualify"""
    for name in LIN_CASES:
        x, P, types, exp = linearity_case(name)
        offs, _ = _layout(types)
        for i, t in enumerate(types):
            if t != 0:
                y = x[offs[i]:offs[i] + 6]
                assert lin_index(F64, x[:3], y, P[offs[i] + 5, offs[i] + 5]) < 0.05, (name, i)
                continue
            y, v = x[offs[i]:offs[i] + 6], P[offs[i] + 5, offs[i] + 5]
            e = lin_index(MP, x[:3], y, v)
            f = lin_index(F64, x[:3], y, v)
            assert abs(abs(e - 0.1) / 0.1 - 1e-9) < 1e-12, (name, i)
            assert abs(f - e) < 1e-13 * 0.1, (name, i)
        assert _first_linear(x, P, types) == exp, name


@pytest.mark.gpu
@pytest.mark.parametrize("name", LIN_CASES)
def test_linearity_choice(name):
    x, P, types, exp = linearity_case(name)
    g = _filter(CAM_R, len(types))
    g.upload_state(x, P, feat_types=types)
    assert g.map_inversedepth_to_cartesian() == exp
    xa, Pa = g.download_state()
    g.close()
    if exp < 0:
        assert np.array_equal(_bits(xa), _bits(x)) and np.array_equal(_bits(Pa), _bits(P))
    # the batched map management picks the same feature (no deletion, no initialisation) and gives the same bits
    gb = _filter(CAM_R, len(types))
    gb.upload_state(x, P, feat_types=types)
    gb.set_image(np.zeros((240, 320), np.uint8))
    rc, status, info = gb.map_management_batch(1, 0, np.zeros((1, 120)))
    assert rc == 0 and list(info[0]) == [0, exp, 0, 0], info
    xb, Pb = gb.download_state()
    assert np.array_equal(_bits(xa), _bits(xb)) and np.array_equal(_bits(Pa), _bits(Pb))


# ---- 4. the new feature's record and patch -----------------------------------------------------------------------------------------
ROWS, COLS, STRIDE = 240, 320, 336
PATCH_UV = [(19.5, 30.0), (20.0, 19.5), (20.75, 20.0), (30.0, 20.75), (19.5, 19.5), (COLS - 1.0, 100.0), (100.0, ROWS - 1.0),
            (COLS - 1.0, ROWS - 1.0), (-30.25, 250.5), (400.0, -50.0), (-0.5, -0.5), (10.2, 5.7)]


def patch_ref(img, rows, cols, ud, vd):
    """cv::Range(ud - 20, ud + 21) with the double bounds truncated toward zero; pixels outside the image read 0"""
    u0, v0 = math.trunc(ud - 20), math.trunc(vd - 20)
    out = np.zeros((41, 41), np.uint8)
    for r in range(41):
        for c in range(41):
            gy, gx = v0 + r, u0 + c
            if 0 <= gx < cols and 0 <= gy < rows:
                out[r, c] = img[gy, gx]
    return out


def test_patch_cases_reach_the_truncation_edges():
    assert {math.trunc(u - 20) != math.floor(u - 20) for u, _ in PATCH_UV} == {True, False}
    assert any(-1 < v - 20 < 0 for _, v in PATCH_UV)


@pytest.mark.gpu
@pytest.mark.parametrize("bound", [True, False])
def test_new_feature_record_and_patch(bound):
    rng = np.random.default_rng(8)
    img = np.full((ROWS, STRIDE), 0xFF, np.uint8)
    img[:, :COLS] = rng.integers(0, 255, (ROWS, COLS))  # 255 only in the padding
    N0 = 4
    x, P, types = _spd_state(N0, 50)
    g = _filter(CAM_R, N0 + len(PATCH_UV))
    g.upload_state(x, P, feat_types=types)
    if bound:
        g.set_image(img, cols=COLS)
    # records of a feature the map forgets: the slot the next addition reuses holds stale counters, flags and patches
    g.set_counters(np.full(N0, 7), np.full(N0, 3))
    g.upload_linearisation(np.ones((N0, 2)), np.ones((N0, 2, 7)), np.ones((N0, 2, 6)), np.ones((N0, 2)), np.ones((N0, 4), np.uint8))
    g.upload_patches(np.full((N0, 13, 13), 9.0))
    g.map_delete_feature(N0 - 1)
    for k, (ud, vd) in enumerate(PATCH_UV):
        n = g.n
        i = g.map_add_feature(np.array([ud, vd]))
        assert i == N0 - 1 + k and list(g.types())[i] == 0 and g.n == n + 6
        xn, _ = g.download_state(want_P=False)
        r = prep_add(F64, xn[:13], CAM_R, ud, vd, 1.0)
        assert _exact_eq(xn[n:n + 6][[0, 1, 2, 5]], _arr(r["xs"])[[0, 1, 2, 5]])  # the feature sits at offset n
        patch, pose = g.feature_init(i)
        want = patch_ref(img, ROWS, COLS, ud, vd) if bound else np.zeros((41, 41), np.uint8)
        assert np.array_equal(patch, want), (ud, vd)
        assert _exact_eq(pose, r["pose14"])
        f = g.features()
        assert f["times_predicted"][i] == 0 and f["times_measured"][i] == 0
        assert not (f["has_h"][i] or f["ic"][i] or f["li"][i] or f["hi"][i])
        assert not g.download_patches()[i].any()
    assert (g.features()["times_predicted"][:N0 - 1] == 7).all()


# ---- 5. FAST-9 ----------------------------------------------------------------------------------------------------------------------
RX = [0, 1, 2, 3, 3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1]
RY = [3, 3, 2, 1, 0, -1, -2, -3, -3, -3, -2, -1, 0, 1, 2, 3]
THRESHOLDS = [0, 1, 99, 100, 101, 254, 255, -5, 300]
TILE = 11


def fast_scores(img, t):
    """plain FAST-9 score of every pixel (0 on the 3-pixel border and for non-corners): best = max over the 16 arcs of 9 of the
    smaller |difference| in one direction; score = best - 1 if best > t"""
    img = np.asarray(img, int)
    H, W = img.shape
    v = img[3:H - 3, 3:W - 3]
    d = np.stack([v - img[3 + dy:H - 3 + dy, 3 + dx:W - 3 + dx] for dx, dy in zip(RX, RY)])
    best = np.full(v.shape, -256)
    for s0 in range(16):
        arc = d[[(s0 + j) % 16 for j in range(9)]]
        best = np.maximum(best, np.maximum(arc.min(0), (-arc).min(0)))
    out = np.zeros(img.shape, int)
    out[3:H - 3, 3:W - 3] = np.where(best > t, best - 1, 0)
    return out


def fast_tiles(t):
    """tiles on a flat background equal to their centre: every arc start, lengths 8, 9, 12, 16, bright and dark arcs of contrast
    t, t + 1, t + 2, centres 0, 128 and 255.  Returns (image, [(cx, cy, length, contrast)])"""
    t = min(max(t, 0), 255)
    specs = []
    for centre in (0, 128, 255):
        for sign in (1, -1):
            for D in (t, t + 1, t + 2):
                val = centre + sign * D
                if D < 1 or not 0 <= val <= 255:
                    continue
                for L in (8, 9, 12, 16):
                    for s in range(16):
                        specs.append((centre, val, L, D, s))
    side = int(math.ceil(math.sqrt(len(specs))))
    img = np.zeros((side * TILE, side * TILE), np.uint8)
    meta = []
    for k, (centre, val, L, D, s) in enumerate(specs):
        y0, x0 = (k // side) * TILE, (k % side) * TILE
        img[y0:y0 + TILE, x0:x0 + TILE] = centre
        cy, cx = y0 + TILE // 2, x0 + TILE // 2
        for j in range(L):
            img[cy + RY[(s + j) % 16], cx + RX[(s + j) % 16]] = val
        meta.append((cx, cy, L, D))
    return img, meta


def _mirror_images(seed=12, S=96):
    """corner-rich noise made symmetric four ways, so that adjacent pixels share a score in every one of the 8 directions"""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, (S, S)).astype(np.uint8)
    lr = np.concatenate([a[:, :S // 2], a[:, :S // 2][:, ::-1]], axis=1)
    ud = np.concatenate([a[:S // 2], a[:S // 2][::-1]], axis=0)
    tr = np.triu(a) + np.triu(a, 1).T
    an = tr[::-1].copy()  # symmetric about the anti-diagonal
    return [lr, ud, tr, an]


def _plateau_dirs(img, t):
    """directions (dx, dy) in which some pixel has a positive score equal to that neighbour's and above its other 7 neighbours'"""
    s = fast_scores(img, t)
    H, W = s.shape
    nb = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if dx or dy]
    found = set()
    for y in range(1, H - 1):
        for x in range(1, W - 1):
            v = s[y, x]
            if v <= 0:
                continue
            eq = [(dx, dy) for dx, dy in nb if s[y + dy, x + dx] == v]
            if len(eq) == 1 and all(s[y + dy, x + dx] < v for dx, dy in nb if (dx, dy) != eq[0]):
                found.add(eq[0])
    return found


def _noise(seed=4, H=120, W=150):
    return np.random.default_rng(seed).integers(0, 256, (H, W)).astype(np.uint8)


FAST_WINDOWS = [(0, 0, 6, 50), (0, 0, 50, 6), (7, 9, 6, 6), (150 - 40, 120 - 30, 40, 30), (13, 17, 41, 25), (3, 9, 41, 50), (0, 0, 150, 120),
                (20, 11, 61, 41)]


def test_fast_designed_tiles_reach_the_edges():
    """every tile's centre scores as designed, including threshold 0 with best = 1 (score 0: no corner, where best itself would be
    one); oracle_py.fast9 agrees with cv2.FAST as a set on these images"""
    import cv2

    for t in THRESHOLDS:
        tc = min(max(t, 0), 255)
        img, meta = fast_tiles(t)
        s = fast_scores(img, tc)
        kinds = set()
        for cx, cy, L, D in meta:
            want = D - 1 if (L >= 9 and D > tc) else 0
            assert s[cy, cx] == want, (t, cx, cy, L, D)
            kinds.add((L, D - tc))
        if tc < 254:
            assert {(L, dd) for L in (8, 9, 12, 16) for dd in (0, 1, 2) if tc + dd >= 1} <= kinds, t
        if tc == 0:
            assert any(D == 1 and L >= 9 for _, _, L, D in meta)
    imgs = [fast_tiles(t)[0] for t in (0, 100, 254)] + _mirror_images() + [_noise()]
    for img in imgs:
        for t in (0, 20, 100):
            ref = {tuple(p) for p in O.fast9(img, t, True, 100000)}
            det = cv2.FastFeatureDetector_create(t, True, cv2.FAST_FEATURE_DETECTOR_TYPE_9_16)
            kp = {(int(k.pt[0]), int(k.pt[1])) for k in det.detect(img)}
            assert ref == kp, t


def test_fast_plateaus_in_every_direction():
    dirs = set()
    for img in _mirror_images():
        dirs |= _plateau_dirs(img, 20)
    assert len(dirs) == 8, dirs


@pytest.mark.gpu
def test_fast9_designed_tiles():
    g = _filter(CAM_R, 4)
    for t in THRESHOLDS:
        img, _ = fast_tiles(t)
        g.set_image(img)
        H, W = img.shape
        kp, n = g.fast_corner_detect_9(0, 0, W, H, t, 100000)
        ref = O.fast9(img, min(max(t, 0), 255), True, 100000)
        assert n == len(ref) and np.array_equal(kp, ref), t


@pytest.mark.gpu
def test_fast9_windows_plateaus_and_max_kp():
    g = _filter(CAM_R, 4)
    img = _noise()
    g.set_image(img)
    for t in (20, 0):
        for x0, y0, w, h in FAST_WINDOWS:
            kp, n = g.fast_corner_detect_9(x0, y0, w, h, t, 100000)
            ref = O.fast9(img[y0:y0 + h, x0:x0 + w], t, True, 100000)
            assert n == len(ref) and np.array_equal(kp, ref), (t, x0, y0, w, h)
            if min(w, h) < 7:
                assert n == 0
    ref = O.fast9(img, 20, True, 100000)
    assert len(ref) > 1100  # the single-CTA compaction runs over many 1024-pixel chunks with keypoints in each
    for max_kp in (1, 7, len(ref) - 1, len(ref)):
        kp, n = g.fast_corner_detect_9(0, 0, img.shape[1], img.shape[0], 20, max_kp)
        assert n == len(ref) and np.array_equal(kp, ref[:max_kp]), max_kp
    for im in _mirror_images():
        g.set_image(im)
        kp, n = g.fast_corner_detect_9(0, 0, im.shape[1], im.shape[0], 20, 100000)
        ref = O.fast9(im, 20, True, 100000)
        assert n == len(ref) and np.array_equal(kp, ref)


# ---- 6. the sampling box -----------------------------------------------------------------------------------------------------------
SX, SY, BAND = 30, 20, 21
DELTA = 2.0**-20  # px, about 1e-6
IMG_B = 1026  # two columns / rows past the camera's 1024, so that boxes reaching the image's right and bottom edge can be cut


def _u_for(c, size, s):
    """the uniform draw that puts the box centre at integer c: cx = round(u (size - 2 band - 2 s)) + band + s"""
    W = size - 2 * BAND - 2 * s
    u = (c - BAND - s) / W
    assert round(u * W) + BAND + s == c
    return u


def box_cases():
    """(name, camera, X, (cx, cy), expected in-box): a cartesian feature X at the identity pose of a dyadic camera"""
    px = lambda cam, hx, hy: np.array([(hx - 512.0) * cam[7], (hy - 512.0) * cam[8], 1.0])  # predicted exactly at (hx, hy)
    cx, cy = 300, 200
    cases = []
    for side, (hx, hy), inward in (("left", (cx - SX, cy), (1, 0)), ("right", (cx + SX, cy), (-1, 0)), ("top", (cx, cy - SY), (0, 1)),
                                   ("bottom", (cx, cy + SY), (0, -1))):
        for tag, k, inside in (("in", 1, True), ("out", -1, False), ("on", 0, False)):
            cases.append((f"{side}-{tag}", CAM_D, px(CAM_D, hx + k * DELTA * inward[0], hy + k * DELTA * inward[1]), (cx, cy), inside))
    tan = lambda a: float(MP.ctx.tan(a))
    third = MP.ctx.pi / 3
    for sgn in (1, -1):
        for tag, eps, vis in (("in", -1e-9, True), ("out", 1e-9, False)):
            X = np.array([sgn * tan(third + eps), 0.01, 1.0])
            cases.append((f"ax{sgn:+d}-{tag}", CAM_D, X, (int(round(512 + 256 * X[0])), 514), vis))
            X = np.array([0.01, sgn * tan(third + eps), 1.0])
            cases.append((f"ay{sgn:+d}-{tag}", CAM_D, X, (514, int(round(512 + 256 * X[1]))), vis))
    for tag, k, vis in (("in", 1, True), ("out", -1, False)):
        cases.append((f"u0-{tag}", CAM_W, px(CAM_W, k * DELTA, 400.0), (SX, 400), vis))
        cases.append((f"v0-{tag}", CAM_W, px(CAM_W, 400.0, k * DELTA), (400, SY), vis))
        cases.append((f"u1-{tag}", CAM_W, px(CAM_W, 1024 - k * DELTA, 400.0), (1024 - SX + 1, 400), vis))
        cases.append((f"v1-{tag}", CAM_W, px(CAM_W, 400.0, 1024 - k * DELTA), (400, 1024 - SY), vis))
    return cases


def _box_image():
    img = np.zeros((IMG_B, IMG_B), np.uint8)
    for cy in range(5, IMG_B - 5, 12):  # a FAST corner every 12 px: centre 0, a bright arc of 12
        for cx in range(5, IMG_B - 5, 12):
            for j in range(12):
                img[cy + RY[j], cx + RX[j]] = 255
    return img


def _box_state(X):
    x = np.r_[0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, np.zeros(6), X]
    return x, np.asfortranarray(np.eye(16) * 1e-4)


def test_box_cases_margins():
    """np_oracle.predict_h (float64) puts every feature on its intended side of the box edge and of the gates, and every window holds
    a FAST corner"""
    img = _box_image()
    for name, cam, X, (cx, cy), inside in box_cases():
        x, _ = _box_state(X)
        h, vis = NP.predict_h(cam, x, [1])
        inb = bool(vis[0]) and cx - SX < h[0, 0] < cx + SX and cy - SY < h[0, 1] < cy + SY
        assert inb == inside, (name, h, vis)
        if name[:2] in ("ax", "ay"):
            hrl = X
            ang = math.degrees(math.atan2(hrl[0] if name[1] == "x" else hrl[1], hrl[2]))
            assert abs(abs(ang) - 60) > 1e-8 and abs(abs(ang) - 60) < 1e-6, name
        elif "-on" not in name and vis[0]:
            edge = min(abs(h[0, 0] - (cx - SX)), abs(h[0, 0] - (cx + SX)), abs(h[0, 1] - (cy - SY)), abs(h[0, 1] - (cy + SY)),
                       abs(h[0, 0]), abs(h[0, 0] - 1024), abs(h[0, 1]), abs(h[0, 1] - 1024))
            assert edge == DELTA, name
        x0, y0 = int(cx - SX), int(cy - SY)
        assert x0 >= 0 and y0 >= 0 and x0 + 2 * SX + 1 <= IMG_B and y0 + 2 * SY + 1 <= IMG_B
        assert len(O.fast9(img[y0:y0 + 2 * SY + 1, x0:x0 + 2 * SX + 1], 100, True)) > 0


@pytest.mark.gpu
def test_sampling_box_edges_and_gates():
    """a feature in the box blocks the attempt (50 attempts, nothing added); one outside lets the window's corner in.  Per-filter
    map_initialize_features, map_management_batch at B = 1 and the C++ oracle's map_management agree with the design"""
    img = _box_image()
    gs = {}
    for name, cam, X, (cx, cy), inside in box_cases():
        if id(cam) not in gs:
            gs[id(cam)] = _filter(cam, 4)
            gs[id(cam)].set_image(img)
        g = gs[id(cam)]
        u = np.tile([_u_for(cx, 1024, SX), _u_for(cy, 1024, SY)], 60)
        want = 0 if inside else 1
        x, P = _box_state(X)
        g.upload_state(x, P, feat_types=[1])
        ni, att = g.map_initialize_features(1, 1, u)
        assert (ni, att) == ((0, 50) if inside else (1, 1)), name
        g.upload_state(x, P, feat_types=[1])
        rc, status, info = g.map_management_batch(1, 1, u[None])
        assert rc == 0 and info[0][2] == want and info[0][3] == (50 if inside else 1), (name, info)
        o = O.OracleFilter(cam)
        o.add_feature(1)
        o.set_state(x, P)
        rco, io = o.map_management(img, 1, 1, u)
        assert rco == 0 and io["initialised"] == want, (name, io)


# ---- 7. k_map_xform past 65535 state rows -------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_add_feature_past_65535_rows():
    """max_features = 10921: N = 10920 gives n = 65533 and n' = 65539 rows, more than one grid dimension's 65535 CTAs.  Needs about
    70 GB of device memory (P and its spare); P is never downloaded"""
    import torch

    free, _ = torch.cuda.mem_get_info(0)
    if free < 80 * 2**30:
        pytest.skip(f"needs 80 GB of free device memory, {free / 2**30:.0f} GB free")
    N = 10920
    rng = np.random.default_rng(9)
    n = 13 + 6 * N
    x = np.zeros(n)
    x[:13] = _camera_x(_q(0.98, 0.05, 0.1, -0.1))
    x[13:] = rng.normal(0, 1, 6 * N)
    g = _filter(CAM_R, N + 1)
    g.upload_state(x, None)
    g.set_image(np.arange(240 * 320, dtype=np.uint64).astype(np.uint8).reshape(240, 320))
    assert g.map_add_feature(np.array([150.25, 100.5])) == N
    assert g.n == n + 6 and g.N == N + 1
    xn, _ = g.download_state(want_P=False)
    r = prep_add(F64, x[:13], CAM_R, 150.25, 100.5, 1.0)
    assert np.array_equal(_bits(xn[:n]), _bits(x)) and _exact_eq(xn[n:][[0, 1, 2, 5]], _arr(r["xs"])[[0, 1, 2, 5]])
    assert (g.types() == 0).all()
    patch, pose = g.feature_init(N)
    img = np.arange(240 * 320, dtype=np.uint64).astype(np.uint8).reshape(240, 320)
    assert np.array_equal(patch, patch_ref(img, 240, 320, 150.25, 100.5)) and _exact_eq(pose, r["pose14"])
    f = g.features()
    assert f["times_predicted"][N] == 0 and not f["has_h"][N]
    g.close()
