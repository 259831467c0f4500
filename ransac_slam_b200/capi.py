"""ctypes binding of the C ABI in include/rslam.h (ransac_slam_b200/lib/librslam_b200.so).

This is plumbing for tests and bench.py; the product is the shared library itself.  There is no CPU fallback: loading
fails loudly if the library has not been built, and every call fails if no CUDA device is present.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSLAM_LIB") or os.path.join(_HERE, "lib", "librslam_b200.so")  # RSLAM_LIB: A/B builds of the same CUDA library during tuning

Q1 = 0x1
Q4 = 0x2
Q6 = 0x4
Q_ALL = 0x7


class RslamError(RuntimeError):
    pass


class Camera(C.Structure):
    _fields_ = [("k1", C.c_double), ("k2", C.c_double), ("nRows", C.c_int), ("nCols", C.c_int), ("Cx", C.c_double), ("Cy", C.c_double),
                ("f", C.c_double), ("dx", C.c_double), ("dy", C.c_double)]


class Params(C.Structure):
    _fields_ = [("std_a", C.c_double), ("std_alpha", C.c_double), ("std_z", C.c_double), ("chi2_095_2", C.c_double),
                ("corr_threshold", C.c_double), ("p_spurious_free", C.c_double), ("n_hyp_initial", C.c_int), ("max_ellipse_eig", C.c_double),
                ("quirks", C.c_uint), ("dedupe_hypotheses", C.c_int)]


class RansacResult(C.Structure):
    _fields_ = [("status", C.c_int), ("hyp_run", C.c_int), ("best_support", C.c_int), ("n_hyp", C.c_int), ("num_ic", C.c_int), ("winner", C.c_int)]


EXPORTS = [
    "rslam_default_params", "rslam_last_error", "rslam_version", "rslam_create", "rslam_destroy", "rslam_sync", "rslam_stream",
    "rslam_launch_count", "rslam_num_features", "rslam_state_dim", "rslam_upload_state", "rslam_download_state", "rslam_upload_patches",
    "rslam_download_features", "rslam_upload_feature_init", "rslam_set_patch_warp", "rslam_download_patches", "rslam_debug_scratch", "rslam_download_H", "rslam_set_matches", "rslam_set_image", "rslam_begin_frame", "rslam_ekf_prediction",
    "rslam_search_ic_matches", "rslam_ransac_hypotheses", "rslam_ransac_result_get", "rslam_update_li", "rslam_rescue_hi", "rslam_update_hi",
    "rslam_frame", "rslam_prefetch_inputs", "rslam_set_graph", "rslam_profile_enable", "rslam_profile_read", "rslam_download_pose", "rslam_support_sweep", "rslam_sweep_mask",
    "rslam_comm_init", "rslam_comm_unique_id", "rslam_comm_init_rank", "rslam_comm_destroy", "rslam_comm_size", "rslam_comm_local_size",
    "rslam_support_sweep_multi", "rslam_upload_linearisation", "rslam_predict_measurements", "rslam_match",
    "rslam_checkpoint_bytes", "rslam_checkpoint_save", "rslam_checkpoint_load",
]

_lib = None


def load():
    """Load the CUDA library.  Raises if it was not built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RslamError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` (no CPU fallback exists)")
    L = C.CDLL(LIB_PATH)
    vp, ci, cd = C.c_void_p, C.c_int, C.c_double
    L.rslam_default_params.argtypes = [C.POINTER(Params)]
    L.rslam_default_params.restype = None
    L.rslam_last_error.restype = C.c_char_p
    L.rslam_version.restype = C.c_char_p
    L.rslam_create.argtypes = [C.POINTER(Camera), C.POINTER(Params), ci, ci, ci, C.POINTER(vp)]
    L.rslam_destroy.argtypes = [vp]
    L.rslam_sync.argtypes = [vp]
    L.rslam_stream.argtypes = [vp]
    L.rslam_stream.restype = vp
    L.rslam_launch_count.argtypes = [vp]
    L.rslam_launch_count.restype = C.c_longlong
    L.rslam_num_features.argtypes = [vp, ci]
    L.rslam_state_dim.argtypes = [vp, ci]
    L.rslam_upload_state.argtypes = [vp, ci, ci, vp, vp, ci, ci, vp, ci]
    L.rslam_download_state.argtypes = [vp, ci, ci, vp, vp, ci]
    L.rslam_upload_patches.argtypes = [vp, ci, vp, ci]
    L.rslam_download_features.argtypes = [vp, ci, vp, vp, vp, vp, vp]
    L.rslam_upload_feature_init.argtypes = [vp, ci, vp, vp, vp, vp, ci]
    L.rslam_set_patch_warp.argtypes = [vp, ci]
    L.rslam_download_patches.argtypes = [vp, ci, vp, ci]
    L.rslam_download_H.argtypes = [vp, ci, vp, vp]
    L.rslam_set_matches.argtypes = [vp, ci, vp, vp]
    L.rslam_upload_linearisation.argtypes = [vp, ci, vp, vp, vp, vp, vp]
    L.rslam_set_image.argtypes = [vp, ci, vp, ci, ci, ci, ci]
    for n in ("rslam_begin_frame", "rslam_ekf_prediction", "rslam_search_ic_matches", "rslam_update_li", "rslam_rescue_hi", "rslam_update_hi", "rslam_predict_measurements",
              "rslam_match"):
        getattr(L, n).argtypes = [vp]
    L.rslam_ransac_hypotheses.argtypes = [vp, vp, ci]
    L.rslam_ransac_result_get.argtypes = [vp, ci, C.POINTER(RansacResult)]
    L.rslam_frame.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci, ci]
    L.rslam_prefetch_inputs.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci]
    L.rslam_download_pose.argtypes = [vp, ci, vp]
    L.rslam_set_graph.argtypes = [vp, ci]
    L.rslam_profile_enable.argtypes = [vp, ci]
    L.rslam_profile_read.argtypes = [vp, C.c_char_p, C.c_size_t]
    L.rslam_support_sweep.argtypes = [vp, vp, ci, ci, ci, ci, ci, vp, vp, vp]
    L.rslam_sweep_mask.argtypes = [vp, ci, vp]
    L.rslam_comm_init.argtypes = [ci, vp, C.POINTER(vp)]
    L.rslam_comm_unique_id.argtypes = [vp]
    L.rslam_comm_init_rank.argtypes = [ci, ci, vp, ci, C.POINTER(vp)]
    L.rslam_comm_destroy.argtypes = [vp]
    L.rslam_comm_size.argtypes = [vp]
    L.rslam_comm_local_size.argtypes = [vp]
    L.rslam_support_sweep_multi.argtypes = [vp, vp, vp, ci, ci, vp, vp, vp]
    L.rslam_map_delete_feature.argtypes = [vp, ci, ci]
    L.rslam_map_delete_features.argtypes = [vp, ci, ci, vp]
    L.rslam_map_inversedepth_to_cartesian.argtypes = [vp, ci, vp]
    L.rslam_map_add_feature.argtypes = [vp, ci, vp, vp]
    L.rslam_fast_corner_detect_9.argtypes = [vp, ci, ci, ci, ci, ci, ci, ci, vp, vp]
    L.rslam_map_initialize_features.argtypes = [vp, ci, ci, ci, vp, ci, vp, vp]
    L.rslam_map_management.argtypes = [vp, ci, ci, ci, ci, vp, ci, vp]
    L.rslam_map_management_batch.argtypes = [vp, ci, ci, ci, vp, ci, vp, vp]
    L.rslam_feature_types.argtypes = [vp, ci, vp]
    L.rslam_set_counters.argtypes = [vp, ci, vp, vp]
    L.rslam_download_feature_init.argtypes = [vp, ci, ci, vp, vp]
    L.rslam_checkpoint_bytes.argtypes = [vp, ci, ci, C.POINTER(C.c_size_t)]
    L.rslam_checkpoint_save.argtypes = [vp, ci, ci, vp, C.c_size_t, C.POINTER(C.c_size_t)]
    L.rslam_checkpoint_load.argtypes = [vp, ci, vp, C.c_size_t, C.POINTER(ci)]
    _lib = L
    return L


def _p(a):
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    return a.ctypes.data_as(C.c_void_p)


def make_camera(cam9):
    c = [float(v) for v in cam9]
    return Camera(c[0], c[1], int(c[2]), int(c[3]), c[4], c[5], c[6], c[7], c[8])


class Filter:
    """A batch of `batch` filters on one GPU (thin wrapper over the opaque rslam_filter handle)."""

    def __init__(self, cam9, max_features, batch=1, device=0, quirks=Q_ALL, std_z=1.0, dedupe=True, n_hyp_initial=1000, std_a=0.007, std_alpha=0.007,
                 max_ellipse_eig=None, p_spurious_free=None):
        self.L = load()
        self.cam = make_camera(cam9)
        self.par = Params()
        self.L.rslam_default_params(C.byref(self.par))
        self.par.quirks = quirks
        self.par.std_z = std_z
        self.par.std_a = std_a
        self.par.std_alpha = std_alpha
        self.par.dedupe_hypotheses = int(dedupe)
        self.par.n_hyp_initial = n_hyp_initial
        if max_ellipse_eig is not None:
            self.par.max_ellipse_eig = max_ellipse_eig
        if p_spurious_free is not None:
            self.par.p_spurious_free = p_spurious_free
        self.h = C.c_void_p()
        self.batch = batch
        self.max_features = max_features
        self._keep = []
        self._ck(self.L.rslam_create(C.byref(self.cam), C.byref(self.par), max_features, batch, device, C.byref(self.h)))

    def _ck(self, rc):
        if rc != 0:
            raise RslamError(f"rslam error {rc}: {self.L.rslam_last_error().decode()}")

    def close(self):
        if self.h:
            self.L.rslam_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- transfers --------------------------------------------------------------------------------------------------
    def upload_state(self, x, P, feat_types=None, b=0, prior=False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = x.size
        ft = None
        if feat_types is None:
            N = (n - 13) // 6
            ft = np.zeros(N, dtype=np.int32)
        else:
            ft = np.ascontiguousarray(feat_types, dtype=np.int32)
            N = ft.size
        if P is not None:
            P = np.asfortranarray(P, dtype=np.float64)
            assert P.shape == (n, n)
        self._ck(self.L.rslam_upload_state(self.h, b, int(prior), _p(x), _p(P), n, n, _p(ft), N))

    def upload_state_device(self, x_ptr, P_ptr, n, ldp, N, b=0, prior=False):
        ft = np.zeros(N, dtype=np.int32)
        self._ck(self.L.rslam_upload_state(self.h, b, int(prior), C.c_void_p(x_ptr), C.c_void_p(P_ptr), n, ldp, _p(ft), N))

    def download_state(self, b=0, prior=False, want_P=True):
        n = self.L.rslam_state_dim(self.h, b)
        x = np.zeros(n)
        P = np.zeros((n, n), order="F") if want_P else None
        self._ck(self.L.rslam_download_state(self.h, b, int(prior), _p(x), _p(P), n))
        return x, P

    def download_pose(self, b=0):
        x = np.zeros(13)
        self._ck(self.L.rslam_download_pose(self.h, b, _p(x)))
        return x

    def upload_patches(self, patches, b=0):
        p = np.ascontiguousarray(patches, dtype=np.float64)
        self._ck(self.L.rslam_upload_patches(self.h, b, _p(p), p.shape[0]))

    def upload_feature_init(self, patches41, r_wc, R_wc, uv, b=0):
        p = np.ascontiguousarray(patches41, dtype=np.uint8)
        r = np.ascontiguousarray(r_wc, dtype=np.float64)
        R = np.ascontiguousarray(R_wc, dtype=np.float64)
        u = np.ascontiguousarray(uv, dtype=np.float64)
        self._ck(self.L.rslam_upload_feature_init(self.h, b, _p(p), _p(r), _p(R), _p(u), p.shape[0]))

    def set_patch_warp(self, enable):
        self._ck(self.L.rslam_set_patch_warp(self.h, int(enable)))

    def download_patches(self, b=0):
        N = self.L.rslam_num_features(self.h, b)
        out = np.zeros((N, 13, 13), dtype=np.float32)
        self._ck(self.L.rslam_download_patches(self.h, b, _p(out), N))
        return out

    def features(self, b=0):
        N = self.L.rslam_num_features(self.h, b)
        h = np.zeros((N, 2))
        S = np.zeros((N, 2, 2))
        z = np.zeros((N, 2))
        flags = np.zeros((N, 4), dtype=np.uint8)
        cnt = np.zeros((N, 2), dtype=np.int32)
        self._ck(self.L.rslam_download_features(self.h, b, _p(h), _p(S), _p(z), _p(flags), _p(cnt)))
        return dict(h=h, S=S, z=z, has_h=flags[:, 0].astype(bool), ic=flags[:, 1].astype(bool), li=flags[:, 2].astype(bool),
                    hi=flags[:, 3].astype(bool), times_predicted=cnt[:, 0], times_measured=cnt[:, 1])

    def H_sparse(self, b=0):
        N = self.L.rslam_num_features(self.h, b)
        Hc = np.zeros((N, 2, 7))
        Hf = np.zeros((N, 2, 6))
        self._ck(self.L.rslam_download_H(self.h, b, _p(Hc), _p(Hf)))
        return Hc, Hf

    def upload_linearisation(self, h, Hc, Hf, z, flags, b=0):
        """Caller-built linearisation of filter b (ExtendKF::update with its own H, z, h): h, z (N, 2); Hc (N, 2, 7); Hf (N, 2, 6), of which
        a cartesian feature uses columns 0..2; flags (N, 4) = has_h, ic, li, hi.  The next update_li / update_hi runs on it."""
        arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (h, Hc, Hf, z)]
        fl = np.ascontiguousarray(flags, dtype=np.uint8)
        self._ck(self.L.rslam_upload_linearisation(self.h, b, *[_p(v) for v in arrs], _p(fl)))

    def set_matches(self, z, ic, b=0):
        z = np.ascontiguousarray(z, dtype=np.float64)
        ic = np.ascontiguousarray(ic, dtype=np.uint8)
        self._ck(self.L.rslam_set_matches(self.h, b, _p(z), _p(ic)))

    def set_image(self, img, b=0, share=False, cols=None):
        """img: uint8 [rows, stride] on the host; the first `cols` (default: all) columns of each row are the image."""
        img = np.ascontiguousarray(img, dtype=np.uint8)
        self._keep = [img]
        cols = img.shape[1] if cols is None else cols
        self._ck(self.L.rslam_set_image(self.h, b, _p(img), img.shape[0], cols, img.shape[1], int(share)))

    # -- stages -----------------------------------------------------------------------------------------------------
    def begin_frame(self):
        self._ck(self.L.rslam_begin_frame(self.h))

    def ekf_prediction(self):
        self._ck(self.L.rslam_ekf_prediction(self.h))

    def search_ic_matches(self):
        self._ck(self.L.rslam_search_ic_matches(self.h))

    def predict_measurements(self):
        self._ck(self.L.rslam_predict_measurements(self.h))

    def match(self):
        self._ck(self.L.rslam_match(self.h))

    def ransac_hypotheses(self, u01, b=0):
        u = np.ascontiguousarray(u01, dtype=np.float64)
        n_u01 = u.size // self.batch
        self._keep = [u]
        self._ck(self.L.rslam_ransac_hypotheses(self.h, _p(u), n_u01))
        return self.ransac_result(b)

    def ransac_result(self, b=0):
        r = RansacResult()
        self._ck(self.L.rslam_ransac_result_get(self.h, b, C.byref(r)))
        return dict(status=r.status, hyp_run=r.hyp_run, best_support=r.best_support, n_hyp=r.n_hyp, num_ic=r.num_ic, winner=r.winner)

    def update_li(self):
        self._ck(self.L.rslam_update_li(self.h))

    def rescue_hi(self):
        self._ck(self.L.rslam_rescue_hi(self.h))

    def update_hi(self):
        self._ck(self.L.rslam_update_hi(self.h))

    def _frame_args(self, images, u01):
        keep = []
        if images is None:
            ip, rows, cols, stride = None, 0, 0, 0
        elif isinstance(images, tuple):
            ip, rows, cols, stride = C.c_void_p(images[0]), images[1], images[2], images[3]
        else:
            img = np.ascontiguousarray(images, dtype=np.uint8)
            rows, cols = img.shape[-2], img.shape[-1]
            stride = cols
            ip = _p(img)
            keep.append(img)
        if isinstance(u01, tuple):
            up, n_u01 = C.c_void_p(u01[0]), u01[1]
        else:
            u = np.ascontiguousarray(u01, dtype=np.float64)
            n_u01 = u.size // self.batch
            up = _p(u)
            keep.append(u)
        return ip, rows, cols, stride, up, n_u01, keep

    def frame(self, images, u01, predict=True, share=False):
        """images: uint8 array [batch, rows, cols] (or [rows, cols] with share) on the host, or (ptr, rows, cols, stride) on the host
        (e.g. pinned memory) or the device.  u01: float64 [batch, n_u01] on the host, or (ptr, n_u01) on the host / device."""
        ip, rows, cols, stride, up, n_u01, keep = self._frame_args(images, u01)
        self._keep = keep
        self._ck(self.L.rslam_frame(self.h, ip, rows, cols, stride, int(share), up, n_u01, 1 if predict else 0))

    def prefetch(self, images, u01, share=False):
        """Start copying the NEXT frame's host inputs (same forms as frame(); (ptr, ...) tuples of pinned memory for an asynchronous
        copy) while the current frame computes; the following frame() with the same host buffers uses them without copying."""
        ip, rows, cols, stride, up, n_u01, keep = self._frame_args(images, u01)
        self._keep_pf = keep
        self._ck(self.L.rslam_prefetch_inputs(self.h, ip, rows, cols, stride, int(share), up, n_u01))

    # ---- Map management (src/Map.cpp), covariance resident on the device ----
    def map_delete_feature(self, index, b=0):
        self._ck(self.L.rslam_map_delete_feature(self.h, b, int(index)))

    def map_delete_features(self, reference_indexing=True, b=0):
        """returns (status, n_deleted); status RSLAM_ERR_REFERENCE_UB (-4) where the reference indexes out of range"""
        nd = C.c_int(0)
        rc = self.L.rslam_map_delete_features(self.h, b, int(reference_indexing), C.byref(nd))
        if rc not in (0, -4):
            self._ck(rc)
        return rc, nd.value

    def map_inversedepth_to_cartesian(self, b=0):
        idx = C.c_int(-1)
        self._ck(self.L.rslam_map_inversedepth_to_cartesian(self.h, b, C.byref(idx)))
        return idx.value

    def map_add_feature(self, uv, b=0):
        uv = np.ascontiguousarray(uv, dtype=np.float64)
        idx = C.c_int(-1)
        self._ck(self.L.rslam_map_add_feature(self.h, b, _p(uv), C.byref(idx)))
        return idx.value

    def fast_corner_detect_9(self, x0=0, y0=0, w=None, h=None, threshold=100, max_kp=4096, b=0):
        """cv::FAST on a window of the bound image; keypoints (x, y) relative to the window, OpenCV order"""
        n = C.c_int(0)
        xy = np.zeros((max_kp, 2), dtype=np.int32)
        self._ck(self.L.rslam_fast_corner_detect_9(self.h, b, x0, y0, w, h, threshold, max_kp, C.byref(n), _p(xy)))
        return xy[: min(n.value, max_kp)].copy(), n.value

    def map_initialize_features(self, step, n, u01, b=0):
        u = np.ascontiguousarray(u01, dtype=np.float64)
        ni, att = C.c_int(0), C.c_int(0)
        self._ck(self.L.rslam_map_initialize_features(self.h, b, int(step), int(n), _p(u), u.size // 2, C.byref(ni), C.byref(att)))
        return ni.value, att.value

    def map_management(self, step, min_features, u01, reference_indexing=True, b=0):
        u = np.ascontiguousarray(u01, dtype=np.float64)
        info = np.zeros(4, dtype=np.int32)
        rc = self.L.rslam_map_management(self.h, b, int(step), int(min_features), int(reference_indexing), _p(u), u.size // 2, _p(info))
        if rc not in (0, -4):
            self._ck(rc)
        return rc, dict(deleted=int(info[0]), converted=int(info[1]), initialised=int(info[2]), attempts=int(info[3]))

    def map_management_batch(self, step, min_features, u01, reference_indexing=True):
        """Map::map_management for every filter at once.  u01: float64 [batch, 2 * n_pairs] on the host (n_pairs >= 50), or
        (device ptr, n_pairs).  Returns (rc, status[batch], info[batch, 4]) with info rows (deleted, converted index or -1,
        initialised, attempts); rc is 0 or the first non-zero status."""
        if isinstance(u01, tuple):
            up, n_pairs = C.c_void_p(u01[0]), int(u01[1])
        else:
            u = np.ascontiguousarray(u01, dtype=np.float64).reshape(self.batch, -1)
            up, n_pairs = _p(u), u.shape[1] // 2
        status = np.zeros(self.batch, dtype=np.int32)
        info = np.zeros((self.batch, 4), dtype=np.int32)
        rc = self.L.rslam_map_management_batch(self.h, int(step), int(min_features), int(reference_indexing), up, n_pairs, _p(status), _p(info))
        if rc not in (0, -3, -4):
            self._ck(rc)
        return rc, status, info

    def types(self, b=0):
        N = self.L.rslam_num_features(self.h, b)
        t = np.zeros(N, dtype=np.int32)
        if N:
            self._ck(self.L.rslam_feature_types(self.h, b, _p(t)))
        return t

    def set_counters(self, times_predicted, times_measured, b=0):
        tp = np.ascontiguousarray(times_predicted, dtype=np.int32)
        tm = np.ascontiguousarray(times_measured, dtype=np.int32)
        self._ck(self.L.rslam_set_counters(self.h, b, _p(tp), _p(tm)))

    def feature_init(self, i, b=0):
        patch = np.zeros((41, 41), dtype=np.uint8)
        pose = np.zeros(14)
        self._ck(self.L.rslam_download_feature_init(self.h, b, int(i), _p(patch), _p(pose)))
        return patch, pose

    # ---- checkpoint / resume (format: include/rslam.h; read_checkpoint below parses it without a GPU) ----
    def checkpoint_bytes(self, b=0, count=None):
        count = self.batch - b if count is None else count
        nb = C.c_size_t(0)
        self._ck(self.L.rslam_checkpoint_bytes(self.h, b, count, C.byref(nb)))
        return nb.value

    def save(self, b=0, count=None, out=None):
        """snapshot of filters [b, b + count) (default: to the end of the batch).  out: None (a new np.uint8 array), a host np.uint8
        array, or a CUDA uint8 tensor on the handle's GPU (saved without host staging).  Returns out[:size] (or the new array)."""
        count = self.batch - b if count is None else count
        if out is None:
            out = np.empty(self.checkpoint_bytes(b, count), dtype=np.uint8)
        written = C.c_size_t(0)
        if isinstance(out, np.ndarray):
            assert out.dtype == np.uint8 and out.flags.c_contiguous
            ptr, cap = _p(out), out.size
        else:  # torch tensor
            assert out.dtype.itemsize == 1 and out.is_contiguous()
            ptr, cap = C.c_void_p(out.data_ptr()), out.numel()
        self._ck(self.L.rslam_checkpoint_save(self.h, b, count, ptr, cap, C.byref(written)))
        return out[: written.value]

    def load(self, buf, b=0):
        """restore every filter of the snapshot buf (np.uint8 array or CUDA uint8 tensor) into slots b, b + 1, ...; returns the count"""
        if isinstance(buf, np.ndarray):
            buf = np.ascontiguousarray(buf, dtype=np.uint8)
            ptr, nb = _p(buf), buf.size
        else:
            assert buf.dtype.itemsize == 1 and buf.is_contiguous()
            ptr, nb = C.c_void_p(buf.data_ptr()), buf.numel()
        cnt = C.c_int(0)
        self._ck(self.L.rslam_checkpoint_load(self.h, b, ptr, nb, C.byref(cnt)))
        return cnt.value

    def set_graph(self, enable):
        self._ck(self.L.rslam_set_graph(self.h, int(enable)))

    def profile(self, enable):
        self._ck(self.L.rslam_profile_enable(self.h, int(enable)))

    def profile_read(self):
        buf = C.create_string_buffer(1 << 16)
        self._ck(self.L.rslam_profile_read(self.h, buf, len(buf)))
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.split()
            out[name] = (int(cnt), float(ms))
        return out

    def sync(self):
        self._ck(self.L.rslam_sync(self.h))

    @property
    def N(self):
        return self.L.rslam_num_features(self.h, 0)

    @property
    def n(self):
        return self.L.rslam_state_dim(self.h, 0)

    @property
    def stream(self):
        return self.L.rslam_stream(self.h)

    @property
    def launches(self):
        return int(self.L.rslam_launch_count(self.h))

    # -- sweep ------------------------------------------------------------------------------------------------------
    def support_sweep(self, hyp_idx, begin=0, end=None, want_mask=True, key_device_ptr=None, n_hyp=None, match_begin=0, match_end=2**31 - 1):
        """hyp_idx: int32 host array or device pointer (int).  Returns (key, mask_bits or None, pairs_scored)."""
        if isinstance(hyp_idx, int):
            hp = C.c_void_p(hyp_idx)
            assert n_hyp is not None
        else:
            hi = np.ascontiguousarray(hyp_idx, dtype=np.int32)
            n_hyp = hi.size
            hp = _p(hi)
            self._keep = [hi]
        end = n_hyp if end is None else end
        key = np.zeros(1, dtype=np.uint64)
        pairs = C.c_longlong(0)
        mask = np.zeros((self.max_features + 7) // 8, dtype=np.uint8) if want_mask else None
        kp = C.c_void_p(key_device_ptr) if key_device_ptr is not None else _p(key)
        self._ck(self.L.rslam_support_sweep(self.h, hp, n_hyp, begin, end, match_begin, match_end, kp, _p(mask), C.byref(pairs) if key_device_ptr is None else None))
        bits = np.unpackbits(mask, bitorder="little").astype(bool) if want_mask else None
        return int(key[0]), bits, int(pairs.value)

    def sweep_mask(self, match_idx):
        mask = np.zeros((self.max_features + 7) // 8, dtype=np.uint8)
        self._ck(self.L.rslam_sweep_mask(self.h, int(match_idx), _p(mask)))
        return np.unpackbits(mask, bitorder="little").astype(bool)


CHECKPOINT_MAGIC = b"RSLAMCKP"
CHECKPOINT_VERSION = 1
_CK_CAMERA = [("k1", "<f8", 24), ("k2", "<f8", 32), ("nRows", "<i4", 40), ("nCols", "<i4", 44), ("Cx", "<f8", 48), ("Cy", "<f8", 56),
              ("f", "<f8", 64), ("dx", "<f8", 72), ("dy", "<f8", 80)]
_CK_PARAMS = [("std_a", "<f8", 88), ("std_alpha", "<f8", 96), ("std_z", "<f8", 104), ("chi2_095_2", "<f8", 112), ("corr_threshold", "<f8", 120),
              ("p_spurious_free", "<f8", 128), ("n_hyp_initial", "<i4", 136), ("max_ellipse_eig", "<f8", 144), ("quirks", "<u4", 152),
              ("dedupe_hypotheses", "<i4", 156)]
# per-filter record arrays after the 16-byte head, in order: (name, dtype, shape per unit, unit "n" or "N")
_CK_RECORDS = [("x", "<f8", (), "n"), ("x_k_km1", "<f8", (), "n"), ("times_predicted", "<i4", (), "N"), ("times_measured", "<i4", (), "N"),
               ("has_h", "u1", (), "N"), ("ic", "u1", (), "N"), ("li", "u1", (), "N"), ("hi", "u1", (), "N"), ("h", "<f8", (2,), "N"),
               ("S", "<f8", (2, 2), "N"), ("z", "<f8", (2,), "N"), ("Hc", "<f8", (2, 7), "N"), ("Hf", "<f8", (2, 6), "N"),
               ("patches", "<f4", (13, 13), "N"), ("patch41", "u1", (41, 41), "N"), ("pose14", "<f8", (14,), "N")]


def _al16(v):
    return (v + 15) & ~15


def read_checkpoint(buf):
    """Parse a snapshot of rslam_checkpoint_save (pure numpy, no GPU).  Returns (header, filters): header = dict(version, count,
    camera=dict, params=dict); filters = list of dicts with n, N, types and the record arrays (x, x_k_km1, counters, flags, h, S, z,
    Hc, Hf, patches, patch41, pose14), and P expanded from the packed lower triangle to the full square."""
    buf = np.frombuffer(bytes(buf) if not isinstance(buf, np.ndarray) else np.ascontiguousarray(buf, dtype=np.uint8).tobytes(), dtype=np.uint8)

    def at(dt, off, count=1):
        return np.frombuffer(buf, dtype=np.dtype(dt), count=count, offset=off)

    if buf.size < 160 or buf[:8].tobytes() != CHECKPOINT_MAGIC:
        raise ValueError("not an rslam snapshot (bad magic)")
    version, count = int(at("<u4", 8)[0]), int(at("<u4", 12)[0])
    total = int(at("<u8", 16)[0])
    if version != CHECKPOINT_VERSION or total != buf.size:
        raise ValueError(f"snapshot version {version}, {total} bytes declared, {buf.size} given")
    header = dict(version=version, count=count, camera={k: at(d, o)[0].item() for k, d, o in _CK_CAMERA},
                  params={k: at(d, o)[0].item() for k, d, o in _CK_PARAMS})
    filters = []
    for i in range(count):
        e = 160 + 32 * i
        boff, toff = int(at("<u8", e)[0]), int(at("<u8", e + 8)[0])
        n, N = int(at("<i4", e + 16)[0]), int(at("<i4", e + 20)[0])
        hn, hN = at("<i4", boff, 2)
        assert (hn, hN) == (n, N), (i, hn, hN, n, N)
        d = dict(n=n, N=N, types=at("<i4", toff, N).copy())
        o = boff + 16
        for name, dt, shape, unit in _CK_RECORDS:
            cnt = (n if unit == "n" else N) * int(np.prod(shape, dtype=np.int64))
            d[name] = at(dt, o, cnt).reshape(((n,) if unit == "n" else (N,) + shape)).copy()
            o += _al16(cnt * np.dtype(dt).itemsize)
        for name in ("has_h", "ic", "li", "hi"):
            d[name] = d[name].astype(bool)
        packed = at("<f8", o, n * (n + 1) // 2)
        P = np.zeros((n, n), order="F")
        j, i = np.triu_indices(n)  # (j, i), i >= j, in row-major order: column j of the lower triangle, rows j..n-1 (LAPACK 'L')
        P[i, j] = packed
        P[j, i] = packed
        d["P"] = P
        filters.append(d)
    return header, filters


def decode_key(key):
    return int(key >> 32), int(0xFFFFFFFF - (key & 0xFFFFFFFF))


SHARD_BY_HYPOTHESIS = 0
SHARD_BY_MATCH = 1


class Comm:
    """NCCL communicator(s) of the sharded sweep, owned by the library (rslam_comm_*)."""

    def __init__(self, handle):
        self.L = load()
        self.h = handle

    @staticmethod
    def _ck(L, rc):
        if rc != 0:
            raise RslamError(f"rslam error {rc}: {L.rslam_last_error().decode()}")

    @classmethod
    def single_process(cls, devices):
        """one host thread driving len(devices) GPUs (ncclCommInitAll)"""
        L = load()
        devs = np.ascontiguousarray(devices, dtype=np.int32)
        h = C.c_void_p()
        cls._ck(L, L.rslam_comm_init(devs.size, _p(devs), C.byref(h)))
        return cls(h)

    @staticmethod
    def unique_id():
        L = load()
        buf = np.zeros(128, dtype=np.uint8)
        Comm._ck(L, L.rslam_comm_unique_id(_p(buf)))
        return buf

    @classmethod
    def from_rank(cls, nranks, rank, uid, device):
        """one process per GPU: uid = the 128 bytes rank 0 obtained from unique_id(), delivered by the caller"""
        L = load()
        uid = np.ascontiguousarray(uid, dtype=np.uint8)
        assert uid.size == 128
        h = C.c_void_p()
        cls._ck(L, L.rslam_comm_init_rank(nranks, rank, _p(uid), device, C.byref(h)))
        return cls(h)

    @property
    def size(self):
        return self.L.rslam_comm_size(self.h)

    @property
    def local_size(self):
        return self.L.rslam_comm_local_size(self.h)

    def support_sweep(self, filters, hyp_idx, shard=SHARD_BY_MATCH, want_mask=True, key_device_ptr=None, n_hyp=None, want_pairs=False):
        """filters: list of Filter (one per local GPU).  hyp_idx: int32 host array or device pointer (int, with n_hyp).
        Returns (key, mask bits or None, pairs scored locally or None); with key_device_ptr the call only enqueues and returns None."""
        arr = (C.c_void_p * len(filters))(*[f.h for f in filters])
        if isinstance(hyp_idx, int):
            hp = C.c_void_p(hyp_idx)
            assert n_hyp is not None
        else:
            hi = np.ascontiguousarray(hyp_idx, dtype=np.int32)
            n_hyp = hi.size
            hp = _p(hi)
            self._keep = hi
        if key_device_ptr is not None:
            self._ck(self.L, self.L.rslam_support_sweep_multi(self.h, arr, hp, n_hyp, shard, C.c_void_p(key_device_ptr), None, None))
            return None
        key = np.zeros(1, dtype=np.uint64)
        pairs = C.c_longlong(0)
        mask = np.zeros((filters[0].max_features + 7) // 8, dtype=np.uint8) if want_mask else None
        self._ck(self.L, self.L.rslam_support_sweep_multi(self.h, arr, hp, n_hyp, shard, _p(key), _p(mask), C.byref(pairs) if want_pairs else None))
        bits = np.unpackbits(mask, bitorder="little").astype(bool) if want_mask else None
        return int(key[0]), bits, (int(pairs.value) if want_pairs else None)

    def close(self):
        if self.h:
            self.L.rslam_comm_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
