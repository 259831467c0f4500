"""ctypes binding of oracle/_ref/libref.so: the reference's OWN hot-path sources (compiled unmodified from /root/reference/src against
the stand-in Eigen / OpenCV / ROS headers of oracle/ref_shim/) behind oracle/ref_driver.cpp.  TEST INFRASTRUCTURE ONLY.

It can be BUILT only where /root/reference exists (the build container: `make -C oracle ref`, done by __graft_entry__.build()); the
GPU box gets the prebuilt, git-ignored .so with the snapshot.  `available()` says whether the library is there; the committed golden
vectors it produced (tests/golden/ref_vectors.*.npz, tests/golden/make_ref_vectors.py) cover the case where it is not.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_ref", "libref.so")
REFERENCE_ROOT = "/root/reference"
RAND_MAX = 2147483647


def build(force=False):
    """(re)build when the reference tree is present; otherwise leave whatever travelled with the snapshot"""
    if not os.path.isdir(os.path.join(REFERENCE_ROOT, "src")):
        return _LIB_PATH if os.path.exists(_LIB_PATH) else None
    if force and os.path.exists(_LIB_PATH):
        os.remove(_LIB_PATH)
    subprocess.check_call(["make", "-C", _HERE, "ref"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


def available():
    return os.path.exists(_LIB_PATH)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError("oracle/_ref/libref.so is missing (it is built from /root/reference by `make -C oracle ref`)")
        L = C.CDLL(_LIB_PATH)
        vp, ci = C.c_void_p, C.c_int
        L.ref_create.restype = vp
        L.ref_create.argtypes = [C.c_char_p]
        for name in ("ref_destroy", "ref_ekf_prediction", "ref_ransac_hypotheses", "ref_update_li", "ref_rescue_hi", "ref_update_hi", "ref_predict_only",
                     "ref_reset_flags"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = None
        for name in ("ref_predict_measurements", "ref_calculate_derivatives"):
            getattr(L, name).argtypes = [vp]
            getattr(L, name).restype = None
        L.ref_S_subset.argtypes = [vp, ci, ci]
        L.ref_ransac_limited.argtypes = [vp, ci]
        L.ref_set_inlier_flags.argtypes = [vp, vp, vp]
        L.ref_set_blocked_gemm.argtypes = [ci, ci]
        L.ref_gemm_seconds.argtypes = [ci, ci, ci]
        L.ref_gemm_seconds.restype = C.c_double
        L.ref_set_rand.argtypes = [vp, ci]
        L.ref_get_camera.argtypes = [vp, vp]
        L.ref_get_params.argtypes = [vp, vp]
        L.ref_track_running.argtypes = [vp, vp, ci, ci, ci]
        L.ref_map_management.argtypes = [vp, vp, ci, ci, ci, ci]
        L.ref_search_ic_matches.argtypes = [vp, vp, ci, ci, ci]
        L.ref_num_features.argtypes = [vp]
        L.ref_state_dim.argtypes = [vp, ci]
        L.ref_get_state.argtypes = [vp, ci, vp, vp]
        L.ref_set_state.argtypes = [vp, ci, vp, vp, ci]
        L.ref_add_feature.argtypes = [vp, ci, vp, vp, vp, vp, vp, ci]
        L.ref_set_counters.argtypes = [vp, vp, vp]
        L.ref_set_matches.argtypes = [vp, vp, vp]
        L.ref_get_features.argtypes = [vp] + [vp] * 6
        L.ref_get_H.argtypes = [vp, ci, vp, ci]
        L.ref_get_patch_matching.argtypes = [vp, ci, vp]
        L.ref_get_feature_init.argtypes = [vp, ci, vp, vp]
        L.ref_distort.argtypes = [vp, vp, ci, vp]
        L.ref_undistort.argtypes = [vp, vp, ci, vp]
        assert L.ref_rand_max() == RAND_MAX
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def set_blocked_gemm(on, threads=1):
    """timing runs only: route the stand-in Eigen's large dense products through the packed kernel of oracle/gemm.cpp"""
    lib().ref_set_blocked_gemm(int(on), int(threads))


def gemm_seconds(m, n, k):
    return float(lib().ref_gemm_seconds(int(m), int(n), int(k)))


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def draws_to_u01(r):
    """the uniforms ExtendKF::rand makes of libc draws r: (double) r / RAND_MAX (src/ExtendKF.cpp:230)"""
    return np.asarray(r, dtype=np.float64) / float(RAND_MAX)


def make_draws(rng, n):
    """n libc-style draws in [0, RAND_MAX) -- RAND_MAX itself is excluded (it would index one past the end, SURVEY A.3 Q8)"""
    return rng.integers(0, RAND_MAX, size=n, dtype=np.int64).astype(np.int32)


YAML_TEMPLATE = """%YAML:1.0
Camera.k1: {k1!r}
Camera.k2: {k2!r}
Camera.nRows: {nRows}
Camera.nCols: {nCols}
Camera.d: {d!r}
Camera.cx_d: {cx_d!r}
Camera.cy_d: {cy_d!r}
Camera.dx: {dx!r}
Camera.dy: {dy!r}
Camera.model: two_distortion_parameters
Camera.fps: {f!r}
Camera.RGB: 1
Sigma.a: {std_a!r}
Sigma.alpha: {std_alpha!r}
Sigma.noise: {std_z!r}
Velocity.v0: {v0!r}
Velocity.stdv0: {std_v0!r}
Velocity.w0: {w0!r}
Velocity.stdw0: {std_w0!r}
min_number_of_features_in_image: {min_features}
"""

# the values of the reference's examples/Monocular/initialize_param.yaml (copied as numbers so that the GPU box, which has no
# /root/reference, can still construct the object)
BUNDLED_YAML = dict(k1=0.06333, k2=0.01390, nRows=240, nCols=320, d=0.0112, cx_d=1.7945, cy_d=1.4433, dx=0.0112, dy=0.0112, f=2.1735,
                    std_a=0.007, std_alpha=0.007, std_z=1.0, v0=0.0, std_v0=0.025, w0=0.00000000001, std_w0=0.025, min_features=25)


class ReferenceFilter:
    """ExtendKF + Map + Tracking of the reference, constructed as System::System does (src/System.cpp:22-70)."""

    def __init__(self, yaml_path=None, tmpdir=None, **overrides):
        self.L = lib()
        if yaml_path is None:
            import tempfile

            vals = dict(BUNDLED_YAML)
            vals.update(overrides)
            fd, yaml_path = tempfile.mkstemp(suffix=".yaml", dir=tmpdir)
            with os.fdopen(fd, "w") as f:
                f.write(YAML_TEMPLATE.format(**vals))
            self._tmp = yaml_path
        else:
            self._tmp = None
        self.h = C.c_void_p(self.L.ref_create(yaml_path.encode()))
        if not self.h:
            raise RuntimeError("reference could not open " + yaml_path)

    def __del__(self):
        try:
            self.L.ref_destroy(self.h)
            if self._tmp:
                os.remove(self._tmp)
        except Exception:
            pass

    # ---- rand queue ----
    def set_draws(self, r):
        r = np.ascontiguousarray(r, dtype=np.int32)
        self.L.ref_set_rand(_p(r), r.size)

    def draws_consumed(self):
        return self.L.ref_rand_consumed()

    def draws_underflow(self):
        return self.L.ref_rand_underflow()

    # ---- parameters ----
    def camera9(self):
        c = np.zeros(9)
        self.L.ref_get_camera(self.h, _p(c))
        return c

    def params(self):
        p = np.zeros(7)
        self.L.ref_get_params(self.h, _p(p))
        return dict(zip(("std_a", "std_alpha", "std_z", "v0", "std_v0", "w0", "std_w0"), p))

    # ---- frame ----
    @staticmethod
    def _img(image):
        return np.ascontiguousarray(image, dtype=np.uint8)

    def track_running(self, image):
        img = self._img(image)
        self.L.ref_track_running(self.h, _p(img), img.shape[0], img.shape[1], img.shape[1])

    def map_management(self, image, step):
        img = self._img(image)
        self.L.ref_map_management(self.h, _p(img), img.shape[0], img.shape[1], img.shape[1], int(step))

    def ekf_prediction(self):
        self.L.ref_ekf_prediction(self.h)

    def search_ic_matches(self, image):
        img = self._img(image)
        self.L.ref_search_ic_matches(self.h, _p(img), img.shape[0], img.shape[1], img.shape[1])

    def predict_only(self):
        self.L.ref_predict_only(self.h)

    # ---- bounded samples of a frame too large to run whole (bench.py, configuration C3) ----
    def predict_measurements(self):
        self.L.ref_predict_measurements(self.h)

    def calculate_derivatives(self):
        self.L.ref_calculate_derivatives(self.h)

    def S_subset(self, first, count):
        return self.L.ref_S_subset(self.h, int(first), int(count))

    def ransac_limited(self, max_hyp):
        return self.L.ref_ransac_limited(self.h, int(max_hyp))

    def set_inlier_flags(self, li, hi):
        li = np.ascontiguousarray(li, dtype=np.uint8)
        hi = np.ascontiguousarray(hi, dtype=np.uint8)
        self.L.ref_set_inlier_flags(self.h, _p(li), _p(hi))

    def reset_flags(self):
        self.L.ref_reset_flags(self.h)

    def ransac_hypotheses(self):
        self.L.ref_ransac_hypotheses(self.h)

    def update_li(self):
        self.L.ref_update_li(self.h)

    def rescue_hi(self):
        self.L.ref_rescue_hi(self.h)

    def update_hi(self):
        self.L.ref_update_hi(self.h)

    # ---- state ----
    @property
    def N(self):
        return self.L.ref_num_features(self.h)

    def n(self, prior=False):
        return self.L.ref_state_dim(self.h, int(prior))

    def get_state(self, prior=False):
        n = self.n(prior)
        x = np.zeros(n)
        P = np.zeros((n, n), order="F")
        self.L.ref_get_state(self.h, int(prior), _p(x), _p(P))
        return x, P

    def set_state(self, x, P, prior=False):
        x = _f64(x)
        P = np.asfortranarray(P, dtype=np.float64)
        assert P.shape == (x.size, x.size)
        self.L.ref_set_state(self.h, int(prior), _p(x), _p(P), x.size)

    def add_feature(self, ftype=0, patch_init=None, patch_match=None, r_wc=None, R_wc=None, uv=None, init_frame=0):
        pi = np.ascontiguousarray(patch_init, dtype=np.uint8) if patch_init is not None else None
        pm = _f64(patch_match) if patch_match is not None else None
        r = _f64(r_wc) if r_wc is not None else None
        R = _f64(R_wc) if R_wc is not None else None
        u = _f64(uv) if uv is not None else None
        self.L.ref_add_feature(self.h, int(ftype), _p(pi), _p(pm), _p(r), _p(R), _p(u), int(init_frame))

    def set_counters(self, times_predicted, times_measured):
        tp = np.ascontiguousarray(times_predicted, dtype=np.int32)
        tm = np.ascontiguousarray(times_measured, dtype=np.int32)
        self.L.ref_set_counters(self.h, _p(tp), _p(tm))

    def set_matches(self, z, ic):
        z = _f64(z)
        ic = np.ascontiguousarray(ic, dtype=np.uint8)
        self.L.ref_set_matches(self.h, _p(z), _p(ic))

    def features(self):
        N = self.N
        h = np.zeros((N, 2))
        S = np.zeros((N, 2, 2))
        z = np.zeros((N, 2))
        flags = np.zeros((N, 4), dtype=np.uint8)
        cnt = np.zeros((N, 2), dtype=np.int32)
        types = np.zeros(N, dtype=np.int32)
        if N:
            self.L.ref_get_features(self.h, _p(h), _p(S), _p(z), _p(flags), _p(cnt), _p(types))
        return dict(h=h, S=S, z=z, has_h=flags[:, 0].astype(bool), ic=flags[:, 1].astype(bool), li=flags[:, 2].astype(bool),
                    hi=flags[:, 3].astype(bool), times_predicted=cnt[:, 0], times_measured=cnt[:, 1], types=types)

    def H_dense(self, i):
        n = self.n(True)
        out = np.zeros((2, n))
        c = self.L.ref_get_H(self.h, int(i), _p(out), n)
        return out[:, :c] if c else None

    def patch_matching(self, i):
        out = np.zeros((13, 13))
        self.L.ref_get_patch_matching(self.h, int(i), _p(out))
        return out

    def feature_init(self, i):
        patch = np.zeros((41, 41), dtype=np.uint8)
        pose = np.zeros(14)
        self.L.ref_get_feature_init(self.h, int(i), _p(patch), _p(pose))
        return patch, pose

    def distort(self, uv):
        uv = _f64(uv).reshape(-1, 2)
        out = np.zeros_like(uv)
        self.L.ref_distort(self.h, _p(uv), uv.shape[0], _p(out))
        return out

    def undistort(self, uv):
        uv = _f64(uv).reshape(-1, 2)
        out = np.zeros_like(uv)
        self.L.ref_undistort(self.h, _p(uv), uv.shape[0], _p(out))
        return out
