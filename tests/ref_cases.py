"""The three cases of tests/golden/ref_vectors.*.npz (produced by the REFERENCE'S OWN SOURCES, see tests/golden/make_ref_vectors.py),
written once against a tiny engine interface so that the CPU oracle and the CUDA path (through the C ABI) are both checked against
the same reference outputs.  Bars (north_star): flags / match indices / hypothesis counts bit-exact, x and P within 1e-9 relative."""
import os

import numpy as np

from tests import golden_npz
from tests import helpers as H

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RAND_MAX = 2147483647


def load():
    return golden_npz.load("ref_vectors")


def u01_of(draws):
    """what ExtendKF::rand (src/ExtendKF.cpp:230) makes of libc draws: (double) r / RAND_MAX"""
    return np.asarray(draws, dtype=np.float64) / float(RAND_MAX)


class OracleEngine:
    """oracle.oracle_py.OracleFilter behind the case interface"""

    name = "oracle"

    def __init__(self, cam9, N_max=64, dense=True):
        from oracle import oracle_py as O

        self.O = O
        self.f = O.OracleFilter(cam9)
        self.f.set_options(O.Q_ALL, sparse=not dense, fast_corr=not dense, warp_patches=True)

    def bootstrap(self, v0, w0, std_v0, std_w0):
        self.f.initialize_x_and_p(v0, w0, std_v0, std_w0)

    def load_map(self, x, P, z):
        for i in range((x.size - 13) // 6):
            self.f.add_feature(0, None, np.zeros((13, 13)), np.zeros(3), np.eye(3), z[i])
        self.f.set_state(x, P, prior=True)
        self.f.set_state(x, P, prior=False)

    def map_management(self, image, step, min_features, u01):
        rc, info = self.f.map_management(image, step, min_features, u01)
        return rc, info["attempts"]

    def ekf_prediction(self):
        self.f.ekf_prediction()

    def search(self, image):
        self.f.search_ic_matches(image)

    def set_matches(self, z, ic):
        self.f.set_matches(z, ic)

    def ransac(self, u01):
        rc, info = self.f.ransac_hypotheses(u01)
        return rc, info["hyp_run"]

    def update_li(self):
        self.f.update_li()

    def rescue_hi(self):
        self.f.rescue_hi()

    def update_hi(self):
        self.f.update_hi()

    def state(self):
        return self.f.get_state()

    def features(self):
        return self.f.features()

    def types(self):
        return self.f.types()

    def init_uv(self):
        return np.array([self.f.feature_init(i)[1][12:] for i in range(self.f.N)])


class GpuEngine:
    """ransac_slam_b200.capi.Filter (the C ABI of librslam_b200.so) behind the case interface"""

    name = "cuda"

    def __init__(self, cam9, N_max=64, dense=True):
        from ransac_slam_b200 import capi

        self.cam9 = cam9
        self.f = capi.Filter(cam9, N_max)
        self.f.set_patch_warp(True)

    def bootstrap(self, v0, w0, std_v0, std_w0):
        # ExtendKF::initialize_x_and_p (src/ExtendKF.cpp:32-54) is host-side set-up: build it here and upload
        eps = np.finfo(np.float64).eps
        x = np.zeros(13)
        x[3] = 1
        x[7:10] = v0
        x[10:13] = w0
        P = np.zeros((13, 13))
        for i in (0, 1, 2, 3, 4, 6):  # index 5 is skipped by the reference (quirk Q7)
            P[i, i] = eps
        for i in (7, 8, 9):
            P[i, i] = std_v0 * std_v0
        for i in (10, 11, 12):
            P[i, i] = std_w0 * std_w0
        self.f.upload_state(x, P, feat_types=np.zeros(0, np.int32))

    def load_map(self, x, P, z):
        N = (x.size - 13) // 6
        self.f.upload_state(x, P, prior=True)
        self.f.upload_state(x, P, prior=False)
        self.f.upload_feature_init(np.zeros((N, 41, 41), np.uint8), np.zeros((N, 3)), np.tile(np.eye(3).reshape(1, 9), (N, 1)), z)

    def map_management(self, image, step, min_features, u01):
        self.f.set_image(image)
        rc, info = self.f.map_management(step, min_features, u01)
        return rc, info["attempts"]

    def ekf_prediction(self):
        self.f.ekf_prediction()

    def search(self, image):
        if image is not None:
            self.f.set_image(image)
        self.f.search_ic_matches()

    def set_matches(self, z, ic):
        self.f.set_matches(z, ic)

    def ransac(self, u01):
        res = self.f.ransac_hypotheses(u01)
        return res["status"], res["hyp_run"]

    def update_li(self):
        self.f.update_li()

    def rescue_hi(self):
        self.f.rescue_hi()

    def update_hi(self):
        self.f.update_hi()

    def state(self):
        return self.f.download_state()

    def features(self):
        return self.f.features()

    def types(self):
        return self.f.types()

    def init_uv(self):
        return np.array([self.f.feature_init(i)[1][12:] for i in range(self.f.N)])


def run_bundled(make_engine, frames=None):
    """System::TrackRunning (src/System.cpp:103-129) over the first frames of the reference's bundled sequence"""
    g = load()
    imgs = np.load(os.path.join(GOLD, "pgm_frames.npz"))["frames"]
    nf = int(g["bundled_frames"]) if frames is None else min(frames, int(g["bundled_frames"]))
    e = make_engine(g["camera9"], 64)
    std_a, std_alpha, std_z, v0, std_v0, w0, std_w0 = g["params7"]
    e.bootstrap(v0, w0, std_v0, std_w0)
    for k in range(nf):
        pre = f"bundled_k{k}_"
        rc, attempts = e.map_management(imgs[k], k + 1, 25, u01_of(g[pre + "draws_map"]))
        assert rc == 0 and 2 * attempts == int(g[pre + "used"][0]), (k, rc, attempts)
        x, P = e.state()
        assert (x.size - 13) // 6 == int(g[pre + "N_before_after"][1])
        assert x.shape == g[pre + "x_map"].shape, (k, x.shape)
        assert list(e.types()) == list(g[pre + "types"])
        assert np.array_equal(e.init_uv(), g[pre + "init_uv"]), f"frame {k}: FAST picked different corners"
        H.assert_x_close(x, g[pre + "x_map"], what=f"{e.name}: x after map_management, frame {k}")
        H.assert_x_close(np.diag(P), g[pre + "Pdiag_map"], what=f"{e.name}: diag P after map_management, frame {k}")
        e.ekf_prediction()
        e.search(imgs[k])
        f = e.features()
        assert np.array_equal(f["has_h"], g[pre + "has_h"]), (k, "has_h")
        assert np.array_equal(f["ic"], g[pre + "ic"]), (k, "ic", f["ic"], g[pre + "ic"])
        ic = g[pre + "ic"]
        assert np.array_equal(f["z"][ic], g[pre + "z"][ic]), (k, "z")
        hh = g[pre + "has_h"]
        np.testing.assert_allclose(f["h"][hh], g[pre + "h"][hh], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(f["S"][hh], g[pre + "S"][hh], rtol=1e-8, atol=1e-9)
        rc, run = e.ransac(u01_of(g[pre + "draws_ransac"]))
        assert rc == 0 and run == int(g[pre + "used"][1]), (k, rc, run)
        assert np.array_equal(e.features()["li"], g[pre + "li"]), (k, "li")
        e.update_li()
        e.rescue_hi()
        assert np.array_equal(e.features()["hi"], g[pre + "hi"]), (k, "hi")
        e.update_hi()
        x, P = e.state()
        H.assert_x_close(x, g[pre + "x"], what=f"{e.name}: x after frame {k}")
        if pre + "P" in g:
            H.assert_P_close(P, g[pre + "P"], what=f"{e.name}: P after frame {k}")
        else:  # later frames store diag(P) and four fixed projections P v instead of the whole matrix
            V = np.random.default_rng(1000 + k).standard_normal((P.shape[0], 4))
            H.assert_x_close(np.diag(P), g[pre + "Pdiag"], what=f"{e.name}: diag P after frame {k}")
            PV, PVg = P @ V, g[pre + "PV"]
            assert np.abs(PV - PVg).max() <= 1e-9 * np.abs(PVg).max() + 1e-12 * np.abs(np.diag(P)).max(), f"{e.name}: P v after frame {k}"
    return nf


def run_q1(make_engine):
    """ransac_hypotheses -> li update -> rescue -> hi update on priors where the bug-compatible support scoring finds inliers"""
    g = load()
    for ci in range(int(g["q1_cases"])):
        pre = f"q1_{ci}_"
        x, P, z, ic = g[pre + "x_in"], g[pre + "P_in"], g[pre + "z"], g[pre + "ic"]
        cam9 = g["camera9"]
        e = make_engine(cam9, (x.size - 13) // 6)
        e.load_map(x, P, z)
        e.search(None)
        f = e.features()
        assert f["has_h"].all()
        np.testing.assert_allclose(f["h"], g[pre + "h"], rtol=1e-12, atol=1e-10)
        np.testing.assert_allclose(f["S"], g[pre + "S"], rtol=1e-9, atol=1e-12)
        e.set_matches(z, ic)
        rc, run = e.ransac(u01_of(g[pre + "draws"]))
        assert rc == 0 and run == int(g[pre + "used"]), (ci, rc, run, int(g[pre + "used"]))
        li = e.features()["li"]
        assert np.array_equal(li, g[pre + "li"]) and li.sum() > 0, (ci, li, g[pre + "li"])
        e.update_li()
        xl, Pl = e.state()
        H.assert_x_close(xl, g[pre + "x_li"], what=f"{e.name}: x after li update, case {ci}")
        H.assert_P_close(Pl, g[pre + "P_li"], what=f"{e.name}: P after li update, case {ci}")
        e.rescue_hi()
        f = e.features()
        assert np.array_equal(f["hi"], g[pre + "hi"]) and f["hi"].sum() > 0, (ci, f["hi"], g[pre + "hi"])
        np.testing.assert_allclose(f["h"], g[pre + "h_rescue"], rtol=1e-12, atol=1e-9)
        e.update_hi()
        xh, Ph = e.state()
        H.assert_x_close(xh, g[pre + "x_hi"], what=f"{e.name}: x after hi update, case {ci}")
        H.assert_P_close(Ph, g[pre + "P_hi"], what=f"{e.name}: P after hi update, case {ci}")


def run_convert(make_engine):
    """Map::map_management with one inverse-depth -> cartesian conversion (src/Map.cpp:105-196) and a blank image"""
    g = load()
    x, P = g["convert_x_in"], g["convert_P_in"]
    N = (x.size - 13) // 6
    e = make_engine(g["camera9"], N + 2)
    e.load_map(x, P, np.zeros((N, 2)))
    blank = np.full((240, 320), 90, np.uint8)
    rc, attempts = e.map_management(blank, 5, 25, u01_of(g["convert_draws"]))
    assert rc == 0 and 2 * attempts == int(g["convert_used"])
    assert list(e.types()) == list(g["convert_types"]) and sum(e.types()) == 1
    xo, Po = e.state()
    H.assert_x_close(xo, g["convert_x"], what=f"{e.name}: x after conversion")
    H.assert_P_close(Po, g["convert_P"], what=f"{e.name}: P after conversion")
    # a whole frame on the mixed map (3- and 6-wide state blocks; calculate_Hi_cartesian, src/Tracking.cpp:71-112)
    e.ekf_prediction()
    e.search(None)
    f = e.features()
    assert np.array_equal(f["has_h"], g["convert_has_h"])
    hh = g["convert_has_h"]
    np.testing.assert_allclose(f["h"][hh], g["convert_h"][hh], rtol=1e-12, atol=1e-10)
    np.testing.assert_allclose(f["S"][hh], g["convert_S"][hh], rtol=1e-9, atol=1e-12)
    e.set_matches(g["convert_z"], g["convert_ic"])
    rc, run = e.ransac(u01_of(g["convert_draws_ransac"]))
    assert rc == 0 and run == int(g["convert_used_ransac"]), (rc, run)
    assert np.array_equal(e.features()["li"], g["convert_li"])
    e.update_li()
    e.rescue_hi()
    assert np.array_equal(e.features()["hi"], g["convert_hi"])
    e.update_hi()
    x2, P2 = e.state()
    H.assert_x_close(x2, g["convert_x_frame"], what=f"{e.name}: x after the frame on the mixed map")
    H.assert_P_close(P2, g["convert_P_frame"], what=f"{e.name}: P after the frame on the mixed map")
