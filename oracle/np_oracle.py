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
