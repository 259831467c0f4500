"""oracle/np_oracle.py -- TEST INFRASTRUCTURE ONLY.  Independent numpy restatement of the algebra of the hot path.

A second opinion for the C++ oracle (oracle/rslam_oracle.cpp): the same reference formulas (SURVEY.md A.1, each function
cites the reference file:line) written directly with numpy / LAPACK, with none of the C++ oracle's code shared.  Used by
tests/ to cross-check the C++ oracle at small N and, because it runs on BLAS, to check the CUDA path at N = 2000 where the
single-threaded dense C++ restatement would take hours.
"""
import numpy as np


def q2r(q):  # src/ExtendKF.cpp:91-102
    r, x, y, z = q
    return np.array([[r * r + x * x - y * y - z * z, 2 * (x * y - r * z), 2 * (z * x + r * y)],
                     [2 * (x * y + r * z), r * r - x * x + y * y - z * z, 2 * (y * z - r * x)],
                     [2 * (z * x - r * y), 2 * (y * z + r * x), r * r - x * x - y * y + z * z]])


def distort_fm(cam, uv):  # src/ExtendKF.cpp:175-204 ; uv: (m, 2)
    k1, k2, _, _, Cx, Cy, _, dx, dy = cam
    xu = (uv[:, 0] - Cx) * dx
    yu = (uv[:, 1] - Cy) * dy
    ru = np.sqrt(xu**2 + yu**2)
    rd = ru / (1 + k1 * ru**2 + k2 * ru**4)
    for _ in range(10):
        f = rd + k1 * rd**3 + k2 * rd**5 - ru
        f_p = 1 + 3 * k1 * rd**2 + 5 * k2 * rd**4
        rd = rd - f / f_p
    D = 1 + k1 * rd**2 + k2 * rd**4
    return np.stack([xu / D / dx + Cx, yu / D / dy + Cy], axis=1)


def jacob_undistor_fm(cam, uvd):  # src/ExtendKF.cpp:312-332
    k1, k2, _, _, Cx, Cy, _, dx, dy = cam
    a, b = uvd[0] - Cx, uvd[1] - Cy
    rd2 = (a * dx) ** 2 + (b * dy) ** 2
    g = k1 + 2 * k2 * rd2
    c = 1 + k1 * rd2 + k2 * rd2 * rd2
    return np.array([[c + a * g * (2 * a * dx * dx), a * g * (2 * b * dy * dy)], [b * g * (2 * a * dx * dx), c + b * g * (2 * b * dy * dy)]])


def dRq_times_a_by_dq(q, a):  # src/ExtendKF.cpp:286-311
    q0, q1, q2, q3 = q
    Ms = [np.array([[q0, -q3, q2], [q3, q0, -q1], [-q2, q1, q0]]), np.array([[q1, q2, q3], [q2, -q1, -q0], [q3, q0, -q1]]),
          np.array([[-q2, q1, q0], [q1, q2, q3], [-q0, q3, -q2]]), np.array([[-q3, -q0, q1], [q0, -q3, q2], [q1, q2, q3]])]
    return np.stack([2 * M @ a for M in Ms], axis=1)


def predict_h(cam, x, types):
    """ExtendKF::predict_camera_measurements + hi_cartesian (src/ExtendKF.cpp:56-132).  Returns h (N,2) and visibility (N,)."""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = cam
    t, R = x[0:3], q2r(x[3:7])
    N = len(types)
    h = np.zeros((N, 2))
    vis = np.zeros(N, bool)
    off = 13
    for i, ty in enumerate(types):
        if ty == 0:
            y = x[off:off + 6]
            m = np.array([np.cos(y[4]) * np.sin(y[3]), -np.sin(y[4]), np.cos(y[4]) * np.cos(y[3])])
            hrl = R.T @ ((y[0:3] - t) * y[5] + m)
            off += 6
        else:
            y = x[off:off + 3]
            hrl = np.linalg.inv(R) @ (y - t)
            off += 3
        ax, ay = np.degrees(np.arctan2(hrl[0], hrl[2])), np.degrees(np.arctan2(hrl[1], hrl[2]))
        if ax < -60 or ax > 60 or ay < -60 or ay > 60:
            continue
        uvu = np.array([[Cx + (hrl[0] / hrl[2]) * f / dx, Cy + (hrl[1] / hrl[2]) * f / dy]])
        uvd = distort_fm(cam, uvu)[0]
        if 0 < uvd[0] < nCols and 0 < uvd[1] < nRows:
            h[i] = uvd
            vis[i] = True
    return h, vis


def jacobian_H(cam, x, types, i, h_i):
    """dense 2 x n H_i (src/Tracking.cpp:71-163)"""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = cam
    n = x.size
    offs = 13 + np.concatenate([[0], np.cumsum([6 if t == 0 else 3 for t in types])])[:-1]
    off = int(offs[i])
    H = np.zeros((2, n))
    a1 = np.linalg.inv(jacob_undistor_fm(cam, h_i))
    Rrw = np.linalg.inv(q2r(x[3:7]))
    r = x[0:3]
    qbar = np.array([x[3], -x[4], -x[5], -x[6]])
    fku, fkv = f / dx, f / dy
    if types[i] == 0:
        y = x[off:off + 6]
        m = np.array([np.cos(y[4]) * np.sin(y[3]), -np.sin(y[4]), np.cos(y[4]) * np.cos(y[3])])
        d = (y[0:3] - r) * y[5] + m
    else:
        y = x[off:off + 3]
        d = y - r
    hc = Rrw @ d
    a2 = np.array([[fku / hc[2], 0, -hc[0] * fku / hc[2] ** 2], [0, fkv / hc[2], -hc[1] * fkv / hc[2] ** 2]])
    A = a1 @ a2
    H[:, 0:3] = A @ (-Rrw) * (y[5] if types[i] == 0 else 1.0)
    H[:, 3:7] = A @ (dRq_times_a_by_dq(qbar, d) @ np.diag([1, -1, -1, -1]))
    if types[i] == 0:
        c2 = np.array([np.cos(y[4]) * np.cos(y[3]), 0, -np.cos(y[4]) * np.sin(y[3])])
        c3 = np.array([-np.sin(y[4]) * np.sin(y[3]), -np.cos(y[4]), -np.sin(y[4]) * np.cos(y[3])])
        c0 = np.column_stack([y[5] * Rrw, Rrw @ c2, Rrw @ c3, Rrw @ (y[0:3] - r)])
        H[:, off:off + 6] = A @ c0
    else:
        H[:, off:off + 3] = A @ Rrw
    return H


def undistort_fm(cam, uv):  # src/ExtendKF.cpp:266-285 ; uv: (m, 2)
    k1, k2, _, _, Cx, Cy, _, dx, dy = cam
    xd = (uv[:, 0] - Cx) * dx
    yd = (uv[:, 1] - Cy) * dy
    rd2 = xd**2 + yd**2
    D = 1 + k1 * rd2 + k2 * rd2**2
    return np.stack([xd * D / dx + Cx, yd * D / dy + Cy], axis=1)


def xyz_w_for_warp(x, types, i):
    """The XYZ_w that Tracking::search_IC_matches hands pred_patch_fc for feature i (src/Tracking.cpp:47-66): the point of the last
    inverse-depth feature at or before i; a cartesian feature does not recompute it (quirk Q3), so one that precedes every
    inverse-depth feature gets the initial zeros."""
    X = np.zeros(3)
    off = 13
    for k in range(i + 1):
        if types[k] == 0:
            y = x[off:off + 6]
            X = y[0:3] + (1.0 / y[5]) * np.array([np.cos(y[4]) * np.sin(y[3]), -np.sin(y[4]), np.cos(y[4]) * np.cos(y[3])])
            off += 6
        else:
            off += 3
    return X


def pred_patch_maps(cam, x, h, XYZ_w, r_init, R_init, uv_init, half_pred=6, half_init=20):
    """Tracking::pred_patch_fc (src/Tracking.cpp:164-278) up to the cv::remap call, for one feature predicted at h (distorted pixel)
    from the prior x: R_init (3 x 3, as uploaded), r_init and uv_init are what Map::initialize_a_features stored, XYZ_w as
    xyz_w_for_warp.  Quirks kept: Q11 (the -1 in the patch offset), Q12 (the translation enters as R r), Q13 (cv::Range truncates).
    Returns (xs, ys, ok, mapx, mapy, c2): the window origin in the current image, ok = -1 if h is within half a patch of the border,
    0 if the truncated window is not 13 x 13 (both give the zero patch), 1 otherwise; mapx / mapy (13 x 13, row = y) are the
    coordinates in the 41 x 41 initial patch that cv::remap samples (None unless ok == 1); c2 is the window centre before truncation
    (None if ok == -1)."""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = cam
    n_len = 2 * half_pred + 1
    if not (half_pred < h[0] < nCols - half_pred and half_pred < h[1] < nRows - half_pred):
        return 0, 0, -1, None, None, None

    def homog4(R, r):  # [R 0; 0 1] [I r; 0 1]
        H4 = np.eye(4)
        H4[:3, :3] = R
        H4[:3, 3] = R @ r
        return H4

    Hpf = homog4(np.asarray(R_init, float).reshape(3, 3), np.asarray(r_init, float))
    Hpfi = np.linalg.inv(Hpf)
    Hkk = Hpfi @ homog4(q2r(x[3:7]), x[0:3])
    n1 = np.array([uv_init[0] - Cx, uv_init[1] - Cy, -f / dx])
    n = n1 / np.linalg.norm(n1)
    nt4 = Hkk @ np.array([h[0] - Cx, h[1] - Cy, -f / dx, 1.0])
    nt = nt4[:3] / nt4[3]
    ns = n + nt / np.linalg.norm(nt)
    n = ns / np.linalg.norm(ns)
    Xk = Hpfi @ np.append(XYZ_w, 1.0)
    d = -(n @ (Xk[:3] / Xk[3]))
    K = np.array([[f / dx, 0, Cx], [0, f / dy, Cy], [0, 0, 1.0]])
    Hm = K @ (Hkk[:3, :3] - np.outer(Hkk[:3, 3], n) / d) @ np.linalg.inv(K)
    w = np.linalg.solve(Hm, np.append(undistort_fm(cam, np.array([uv_init]))[0], 1.0))
    c2 = distort_fm(cam, np.array([w[:2] / w[2]]))[0]
    xs, xe = int(c2[0] - half_pred), int(c2[0] + half_pred)  # int() truncates toward zero like cv::Range(double, double)
    ys, ye = int(c2[1] - half_pred), int(c2[1] + half_pred)
    if xe - xs + 1 != n_len or ye - ys + 1 != n_len:
        return xs, ys, 0, None, None, c2
    gy, gx = np.mgrid[ys:ys + n_len, xs:xs + n_len].astype(float)
    und = undistort_fm(cam, np.stack([gx.ravel(), gy.ravel()], axis=1))
    p = Hm @ np.vstack([und.T, np.ones(und.shape[0])])
    with np.errstate(divide="ignore", invalid="ignore"):
        c1 = distort_fm(cam, np.stack([p[0] / p[2], p[1] / p[2]], axis=1))
    mapx = c1[:, 0].reshape(n_len, n_len) - (uv_init[0] - half_init - 1)
    mapy = c1[:, 1].reshape(n_len, n_len) - (uv_init[1] - half_init - 1)
    return xs, ys, 1, mapx, mapy, c2


def v2q(v, eps=2.220446049250313e-16):  # src/ExtendKF.cpp:428-443 (quirk Q14: the zero quaternion below eps)
    theta = np.sqrt(v @ v)
    if theta < eps:
        return np.zeros(4)
    vn = v / theta
    return np.concatenate([[np.cos(theta / 2.0)], np.sin(theta / 2.0) * (vn / np.sqrt(vn @ vn))])


def qprod(q, p):  # src/ExtendKF.cpp:416-427: q * p with the vector part (q0 p_v + p0 q_v) + q_v x p_v
    return np.concatenate([[q[0] * p[0] - q[1:] @ p[1:]], q[0] * p[1:] + p[0] * q[1:] + np.cross(q[1:], p[1:])])


def dq3_by_dq1(q):  # src/ExtendKF.cpp:482-490
    return np.array([[q[0], -q[1], -q[2], -q[3]], [q[1], q[0], -q[3], q[2]], [q[2], q[3], q[0], -q[1]], [q[3], -q[2], q[1], q[0]]])


def dqomegadt_by_domega(w, dt=1.0):  # src/ExtendKF.cpp:491-529
    om = np.sqrt(w @ w)
    s, c = np.sin(om * dt / 2.0), np.cos(om * dt / 2.0)
    m = np.zeros((4, 3))
    m[0] = (-dt / 2.0) * (w / om) * s
    for i in range(3):
        for j in range(3):
            if i == j:
                m[1 + i, j] = (dt / 2.0) * w[i] * w[i] / (om * om) * c + (1.0 / om) * (1.0 - w[i] * w[i] / (om * om)) * s
            else:
                m[1 + i, j] = (w[i] * w[j] / (om * om)) * ((dt / 2.0) * c - (1.0 / om) * s)
    return m


def ekf_prediction(x, P, std_a, std_alpha, dt=1.0):
    """ExtendKF::ekf_prediction (src/ExtendKF.cpp:333-388), constant velocity: x_k_km1 = [fv(x_v); y] and
    P_k_km1 = [F P_cc F^T + Q, F P_cf; P_fc F^T, P_ff] with F = dfv_by_dxv (:444-481) and Q = G diag(la, la, la, aa, aa, aa) G^T
    (:347-376).  Returns (x_k_km1, P_k_km1)."""
    x = np.asarray(x, dtype=np.float64)
    qwt = v2q(x[10:13] * dt)
    xv = np.concatenate([x[0:3] + x[7:10] * dt, qprod(x[3:7], qwt), x[7:13]])  # fv
    F = np.eye(13)
    F[0:3, 7:10] = dt * np.eye(3)
    F[3:7, 3:7] = np.array([[qwt[0], -qwt[1], -qwt[2], -qwt[3]], [qwt[1], qwt[0], qwt[3], -qwt[2]], [qwt[2], -qwt[3], qwt[0], qwt[1]],
                            [qwt[3], qwt[2], -qwt[1], qwt[0]]])  # d(q * qwt) / dq, in dfv_by_dxv (:444-481)
    ab = dq3_by_dq1(x[3:7]) @ dqomegadt_by_domega(x[10:13], dt)
    F[3:7, 10:13] = ab
    G = np.zeros((13, 6))
    G[0:3, 0:3] = dt * np.eye(3)
    G[3:7, 3:6] = ab
    G[7:10, 0:3] = np.eye(3)
    G[10:13, 3:6] = np.eye(3)
    Q = G @ np.diag([(std_a * dt) ** 2] * 3 + [(std_alpha * dt) ** 2] * 3) @ G.T
    xo = x.copy()
    xo[0:13] = xv
    Po = np.array(P, dtype=np.float64, order="F", copy=True)
    Po[0:13, 0:13] = F @ P[0:13, 0:13] @ F.T + Q
    Po[0:13, 13:] = F @ P[0:13, 13:]
    Po[13:, 0:13] = P[13:, 0:13] @ F.T
    return xo, Po


def ekf_update(x, P, H, z, h, q4_int_exponent=True):
    """ExtendKF::update (src/ExtendKF.cpp:597-639), dense, general inverse."""
    if z.size == 0:
        return x.copy(), P.copy()
    k = z.size
    S = H @ P @ H.T + np.eye(k)
    K = P @ H.T @ np.linalg.inv(S)
    xkk = x + K @ (z - h)
    Pt = P - K @ S @ K.T
    Pk = 0.5 * Pt + 0.5 * Pt.T
    return normalise_quaternion(xkk, Pk, q4_int_exponent)


def normalise_quaternion(xkk, Pk, q4_int_exponent=True):
    """The quaternion normalisation that closes ExtendKF::update (src/ExtendKF.cpp:611-634): x_k_k[3:7] / |q| and
    P <- Tm P Tm^T with Tm the identity except for Jn in rows / columns 3..6.  Tm is applied to those four rows and columns only
    (O(n) instead of two dense n^3 products)."""
    r, qx, qy, qz = xkk[3:7]
    s = r * r + qx * qx + qy * qy + qz * qz
    T = np.array([[qx * qx + qy * qy + qz * qz, -r * qx, -r * qy, -r * qz], [-qx * r, r * r + qy * qy + qz * qz, -qx * qy, -qx * qz],
                  [-qy * r, -qy * qx, r * r + qx * qx + qz * qz, -qy * qz], [-qz * r, -qz * qx, -qz * qy, r * r + qx * qx + qy * qy]])
    Jn = (s ** -1.0 if q4_int_exponent else s ** -1.5) * T
    xkk = xkk.copy()
    xkk[3:7] = xkk[3:7] / np.sqrt(s)
    Pn = np.array(Pk, copy=True)
    Pn[3:7, :] = Jn @ Pn[3:7, :]
    Pn[:, 3:7] = Pn[:, 3:7] @ Jn.T
    return xkk, Pn


def hypothesis_support(cam, x, P, types, H_p, h_p, z_p, z_all, has_z, std_z=1.0, q1=True):
    """One 1-point hypothesis + support (src/Tracking.cpp:419-477).  z_all (N,2); has_z (N,) ; inverse-depth features only.
    returns (support, inlier mask over matched features, residuals)."""
    k1, k2, nRows, nCols, Cx, Cy, f, dx, dy = cam
    S = H_p @ P @ H_p.T + np.eye(2)
    K = P @ H_p.T @ np.linalg.inv(S)
    xi = x + K @ (z_p - h_p)
    offs = 13 + 6 * np.arange(len(types))
    mo = offs[has_z]
    m = mo.size
    ri_v = np.concatenate([xi[o:o + 3] for o in mo]) if m else np.zeros(0)
    ang_v = np.concatenate([xi[o + 3:o + 5] for o in mo]) if m else np.zeros(0)
    rho = np.array([xi[o + 5] for o in mo])
    src = ri_v if q1 else ang_v
    a0, a1 = src[0:2 * m:2], src[1:2 * m:2]
    mi = np.stack([np.cos(a1) * np.sin(a0), -np.sin(a1), np.cos(a1) * np.cos(a0)], axis=0)
    ri = ri_v.reshape(m, 3).T
    v = (ri - xi[0:3, None]) * rho[None, :] + mi
    hc = q2r(xi[3:7]).T @ v
    himg = np.stack([f / dx * hc[0] / hc[2] + Cx, f / dx * hc[1] / hc[2] + Cy], axis=1)
    hd = distort_fm(cam, himg)
    res = np.sqrt(((z_all[has_z] - hd) ** 2).sum(axis=1))
    inl = res < std_z
    return int(inl.sum()), inl, res
