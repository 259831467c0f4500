"""ctypes binding of the CPU oracle (oracle/_build/liborc.so).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
The product package ransac_slam_b200 never does (tests/test_no_oracle_in_product.py enforces it).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "liborc.so")
_SHIM_PATH = os.path.join(_HERE, "_build", "libshim.so")

Q1 = 1 << 0  # angles taken from the position vector (src/Tracking.cpp:448)
Q4 = 1 << 1  # pow(s, -3/2) -> s^-1 (src/ExtendKF.cpp:627)
Q6 = 1 << 2  # rescue gate without +R (src/Tracking.cpp:589)
Q11 = 1 << 3  # MATLAB -1 offset kept in the remap coordinates (src/Tracking.cpp:264-265)
Q_ALL = 0xF


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("rslam_oracle.cpp", "gemm.cpp", "omat.h", "shim_probe.cpp", "ref_shim/mini_eigen.h", "ref_shim/mini_cv.h",
                                             "Makefile")]
    if (not force) and all(os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(s) for s in srcs) for out in (_LIB_PATH, _SHIM_PATH)):
        return _LIB_PATH
    subprocess.check_call(["make", "-C", _HERE, "all"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_LIB_PATH)
        _lib.orc_create.restype = C.c_void_p
        _lib.orc_create.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double]
        for name in ("orc_destroy", "orc_map_reset_flags", "orc_ekf_prediction", "orc_update_li", "orc_rescue_hi", "orc_update_hi"):
            getattr(_lib, name).argtypes = [C.c_void_p]
            getattr(_lib, name).restype = None
        _lib.orc_set_options.argtypes = [C.c_void_p, C.c_uint, C.c_int, C.c_int, C.c_int]
        _lib.orc_set_threads.argtypes = [C.c_int]
        _lib.orc_num_features.argtypes = [C.c_void_p]
        _lib.orc_state_dim.argtypes = [C.c_void_p]
        _lib.orc_set_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        _lib.orc_get_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        _lib.orc_add_feature.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 5
        _lib.orc_set_patch_matching.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_get_patch_matching.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_set_matches.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_search_ic_matches.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        _lib.orc_ransac_hypotheses.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        _lib.orc_ransac_info.argtypes = [C.c_void_p, C.c_void_p]
        _lib.orc_get_features.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        _lib.orc_get_H.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_cv_remap.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _lib.orc_corrcoef.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _lib.orc_distort.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_undistort.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_lu_inverse.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_dgemm.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        _lib.orc_fast9.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        _lib.orc_initialize_features.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_map_management.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_initialize_x_and_p.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double]
        _lib.orc_map_delete_pass.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        _lib.orc_map_delete_feature.argtypes = [C.c_void_p, C.c_int]
        _lib.orc_map_inversedepth_to_cartesian.argtypes = [C.c_void_p]
        _lib.orc_map_add_feature.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        _lib.orc_set_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_get_types.argtypes = [C.c_void_p, C.c_void_p]
        _lib.orc_get_feature_init.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return _lib


def shim_lib():
    """oracle/_build/libshim.so: the stand-in Eigen / OpenCV headers of ref_shim/ behind C entry points (shim_probe.cpp)"""
    build()
    return C.CDLL(_SHIM_PATH)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class OracleFilter:
    """One EKF filter in the oracle.  cam = (k1,k2,nRows,nCols,Cx,Cy,f,dx,dy)."""

    def __init__(self, cam9, std_a=0.007, std_alpha=0.007, std_z=1.0, quirks=Q_ALL, sparse=False, fast_corr=False, warp_patches=False):
        self.L = lib()
        cam = _f64(cam9)
        self.h = C.c_void_p(self.L.orc_create(_p(cam), std_a, std_alpha, std_z))
        self.L.orc_set_options(self.h, quirks, int(sparse), int(fast_corr), int(warp_patches))

    def __del__(self):
        try:
            self.L.orc_destroy(self.h)
        except Exception:
            pass

    def set_options(self, quirks=Q_ALL, sparse=False, fast_corr=False, warp_patches=False):
        self.L.orc_set_options(self.h, quirks, int(sparse), int(fast_corr), int(warp_patches))

    @property
    def N(self):
        return self.L.orc_num_features(self.h)

    @property
    def n(self):
        return self.L.orc_state_dim(self.h)

    def add_feature(self, ftype=0, patch_init=None, patch_match=None, r_wc=None, R_wc=None, uv=None):
        pi = np.ascontiguousarray(patch_init, dtype=np.uint8) if patch_init is not None else None
        pm = _f64(patch_match) if patch_match is not None else None
        r = _f64(r_wc) if r_wc is not None else None
        R = _f64(R_wc) if R_wc is not None else None
        u = _f64(uv) if uv is not None else None
        return self.L.orc_add_feature(self.h, int(ftype), _p(pi), _p(pm), _p(r), _p(R), _p(u))

    def set_state(self, x, P, prior=False):
        x = _f64(x)
        P = np.asfortranarray(P, dtype=np.float64)
        assert P.shape == (x.size, x.size)
        self.L.orc_set_state(self.h, int(prior), _p(x), _p(P), x.size)

    def get_state(self, prior=False, want_P=True):
        n = self.n
        x = np.zeros(n)
        P = np.zeros((n, n), order="F") if want_P else None
        self.L.orc_get_state(self.h, int(prior), _p(x), _p(P))
        return x, P

    def set_matches(self, z, ic):
        z = _f64(z)
        ic = np.ascontiguousarray(ic, dtype=np.uint8)
        self.L.orc_set_matches(self.h, _p(z), _p(ic))

    def map_reset_flags(self):
        self.L.orc_map_reset_flags(self.h)

    def ekf_prediction(self):
        self.L.orc_ekf_prediction(self.h)

    def search_ic_matches(self, image=None):
        if image is None:
            self.L.orc_search_ic_matches(self.h, None, 0, 0, 0)
        else:
            img = np.ascontiguousarray(image, dtype=np.uint8)
            self.L.orc_search_ic_matches(self.h, _p(img), img.shape[0], img.shape[1], img.shape[1])

    def ransac_hypotheses(self, u01):
        u = _f64(u01)
        rc = self.L.orc_ransac_hypotheses(self.h, _p(u), u.size)
        info = np.zeros(4, dtype=np.int32)
        self.L.orc_ransac_info(self.h, _p(info))
        return rc, dict(hyp_run=int(info[0]), best_support=int(info[1]), n_hyp=int(info[2]), num_ic=int(info[3]))

    def update_li(self):
        self.L.orc_update_li(self.h)

    def rescue_hi(self):
        self.L.orc_rescue_hi(self.h)

    def update_hi(self):
        self.L.orc_update_hi(self.h)

    def features(self):
        N = self.N
        h = np.zeros((N, 2))
        S = np.zeros((N, 2, 2))
        z = np.zeros((N, 2))
        flags = np.zeros((N, 4), dtype=np.uint8)
        cnt = np.zeros((N, 2), dtype=np.int32)
        self.L.orc_get_features(self.h, _p(h), _p(S), _p(z), _p(flags), _p(cnt))
        return dict(h=h, S=S, z=z, has_h=flags[:, 0].astype(bool), ic=flags[:, 1].astype(bool), li=flags[:, 2].astype(bool),
                    hi=flags[:, 3].astype(bool), times_predicted=cnt[:, 0], times_measured=cnt[:, 1])

    def H_dense(self, i):
        out = np.zeros((2, self.n))
        self.L.orc_get_H(self.h, int(i), _p(out))
        return out

    def patch_matching(self, i):
        out = np.zeros((13, 13))
        self.L.orc_get_patch_matching(self.h, int(i), _p(out))
        return out

    def distort(self, uv):
        uv = _f64(uv).reshape(-1, 2)
        out = np.zeros_like(uv)
        self.L.orc_distort(self.h, _p(uv), uv.shape[0], _p(out))
        return out

    def undistort(self, uv):
        uv = _f64(uv).reshape(-1, 2)
        out = np.zeros_like(uv)
        self.L.orc_undistort(self.h, _p(uv), uv.shape[0], _p(out))
        return out

    # ---- Map management (src/Map.cpp) ----
    def map_delete_pass(self, reference_indexing=True):
        """Map::map_management step 1 (src/Map.cpp:19-32); returns (status, n_deleted); status -4 = the reference reads out of range"""
        nd = C.c_int(0)
        rc = self.L.orc_map_delete_pass(self.h, int(reference_indexing), C.byref(nd))
        return rc, nd.value

    def map_delete_feature(self, index):
        return self.L.orc_map_delete_feature(self.h, int(index))

    def map_inversedepth_to_cartesian(self):
        """Map::inversedepth_2_cartesian (src/Map.cpp:105-196); returns the converted feature index or -1"""
        return self.L.orc_map_inversedepth_to_cartesian(self.h)

    def map_add_feature(self, uv, image=None):
        """hinv + add_a_feature_covariance_inverse_depth + features_info.push_back (src/Map.cpp:268-311, 339-400)"""
        uv = _f64(uv)
        if image is None:
            return self.L.orc_map_add_feature(self.h, _p(uv), None, 0, 0, 0)
        img = np.ascontiguousarray(image, dtype=np.uint8)
        return self.L.orc_map_add_feature(self.h, _p(uv), _p(img), img.shape[0], img.shape[1], img.shape[1])

    def initialize_x_and_p(self, v0=0.0, w0=1e-11, std_v0=0.025, std_w0=0.025):
        """ExtendKF::initialize_x_and_p (src/ExtendKF.cpp:32-54) with the yaml's Velocity.* values"""
        self.L.orc_initialize_x_and_p(self.h, v0, w0, std_v0, std_w0)

    def initialize_features(self, step, n, image, u01):
        """Map::initialize_features (src/Map.cpp:198-211); u01: 2 draws per attempt.  Returns (initialised or -1, attempts)"""
        img = np.ascontiguousarray(image, dtype=np.uint8)
        u = _f64(u01)
        att = C.c_int(0)
        r = self.L.orc_initialize_features(self.h, int(step), int(n), _p(img), img.shape[0], img.shape[1], img.shape[1], _p(u), u.size // 2, C.byref(att))
        return r, att.value

    def map_management(self, image, step, min_features, u01, reference_indexing=True):
        """Map::map_management (src/Map.cpp:16-67).  Returns (status, dict(deleted, converted, initialised, attempts))"""
        img = np.ascontiguousarray(image, dtype=np.uint8)
        u = _f64(u01)
        info = np.zeros(4, dtype=np.int32)
        rc = self.L.orc_map_management(self.h, _p(img), img.shape[0], img.shape[1], img.shape[1], int(step), int(min_features), int(reference_indexing), _p(u),
                                       u.size // 2, _p(info))
        return rc, dict(deleted=int(info[0]), converted=int(info[1]), initialised=int(info[2]), attempts=int(info[3]))

    def set_counters(self, times_predicted, times_measured):
        tp = np.ascontiguousarray(times_predicted, dtype=np.int32)
        tm = np.ascontiguousarray(times_measured, dtype=np.int32)
        self.L.orc_set_counters(self.h, _p(tp), _p(tm))

    def types(self):
        t = np.zeros(self.N, dtype=np.int32)
        if self.N:
            self.L.orc_get_types(self.h, _p(t))
        return t

    def feature_init(self, i):
        patch = np.zeros((41, 41), dtype=np.uint8)
        pose = np.zeros(14)
        self.L.orc_get_feature_init(self.h, int(i), _p(patch), _p(pose))
        return patch, pose

    def frame(self, image, u01, predict=True):
        """One TrackRunning pass (src/System.cpp:111-129) without Map feature add/delete."""
        if predict:
            self.map_reset_flags()
            self.ekf_prediction()
        self.search_ic_matches(image)
        rc, info = self.ransac_hypotheses(u01)
        self.update_li()
        self.rescue_hi()
        self.update_hi()
        return rc, info


def fast9(image, threshold=100, nonmax=True, max_kp=4096):
    """cv::FAST restatement (src/Map.cpp:324-338 calls cv::FAST(im, kps, 100, true)); returns keypoints (x, y) in OpenCV's order"""
    img = np.ascontiguousarray(image, dtype=np.uint8)
    xy = np.zeros((max_kp, 2), dtype=np.int32)
    n = lib().orc_fast9(_p(img), img.shape[0], img.shape[1], img.shape[1], int(threshold), int(nonmax), max_kp, _p(xy))
    return xy[: min(n, max_kp)].copy()


def cv_remap(src, mapx, mapy):
    src = _f64(src)
    mapx = _f64(mapx)
    mapy = _f64(mapy)
    out = np.zeros(mapx.shape)
    lib().orc_cv_remap(_p(src), src.shape[0], src.shape[1], _p(mapx), _p(mapy), mapx.shape[0], mapx.shape[1], _p(out))
    return out


def corrcoef(M, row0_only=False):
    M = _f64(M)
    out = np.zeros((M.shape[1], M.shape[1]))
    lib().orc_corrcoef(_p(M), M.shape[0], M.shape[1], int(row0_only), _p(out))
    return out


def lu_inverse(A):
    A = np.asfortranarray(A, dtype=np.float64)
    out = np.zeros_like(A, order="F")
    lib().orc_lu_inverse(_p(A), A.shape[0], _p(out))
    return out


def dgemm(A, B, tA=False, tB=False):
    A = np.asfortranarray(A, dtype=np.float64)
    B = np.asfortranarray(B, dtype=np.float64)
    M = A.shape[1] if tA else A.shape[0]
    K = A.shape[0] if tA else A.shape[1]
    N = B.shape[0] if tB else B.shape[1]
    Cm = np.zeros((M, N), order="F")
    lib().orc_dgemm(int(tA), int(tB), M, N, K, _p(A), A.shape[0], _p(B), B.shape[0], _p(Cm), M)
    return Cm


def set_threads(n):
    lib().orc_set_threads(int(n))
