"""Generates tests/golden/ref_vectors.*.npz from the REFERENCE'S OWN SOURCES (oracle/_ref/libref.so = /root/reference/src/{ExtendKF,
Tracking,Converter,Map}.cpp compiled unmodified against the stand-in third-party headers of oracle/ref_shim/, see
oracle/ref_driver.cpp).  Run in the build container, where /root/reference exists:

    make -C oracle ref && python tests/golden/make_ref_vectors.py

The GPU box has no /root/reference; there the tests read this .npz (and use the prebuilt libref.so if it travelled).

Case "bundled": the first frames of the reference's bundled sequence (tests/golden/pgm_frames.npz) through the whole
System::TrackRunning call sequence (src/System.cpp:103-129), libc rand() fed from a recorded queue.
Case "q1": a synthetic prior on which the reference's (bug-compatible) support scoring finds real inliers
(tests/helpers.py:q1_consistent_state), through ransac_hypotheses / li update / rescue / hi update.
Case "convert": Map::map_management on a map whose first feature passes the linearity test (src/Map.cpp:105-196).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_py as R  # noqa: E402
from tests import golden_npz  # noqa: E402
from tests import helpers as H  # noqa: E402

BUNDLED_FRAMES = 9          # frames 7 and 8 run Map::map_management's delete pass (12 and 8 deletions, run-ahead index, src/Map.cpp:19-32)
BUNDLED_FULL_P = 6          # full covariance stored for the first frames, diag + 4 fixed projections P v afterwards (file size)
Q1_CASES = [(20, 3, 0.2), (16, 8, 0.45)]  # (N, seed, outlier fraction)


def bundled(out):
    p = np.load(os.path.join(ROOT, "tests", "golden", "pgm_frames.npz"))
    frames = p["frames"]
    r = R.ReferenceFilter()
    out["camera9"] = r.camera9()
    out["params7"] = np.array(list(r.params().values()))
    rng = np.random.default_rng(11)
    for k in range(BUNDLED_FRAMES):
        dm = R.make_draws(rng, 200)
        dr = R.make_draws(rng, 1000)
        n_before = r.N
        r.set_draws(dm)
        r.map_management(frames[k], k + 1)
        used_m = r.draws_consumed()
        x_map, P_map = r.get_state()
        f_map = r.features()
        r.ekf_prediction()
        r.search_ic_matches(frames[k])
        f_s = r.features()
        r.set_draws(dr)
        r.ransac_hypotheses()
        used_r = r.draws_consumed()
        assert r.draws_underflow() == 0
        f_r = r.features()
        r.update_li()
        r.rescue_hi()
        f_h = r.features()
        r.update_hi()
        x, P = r.get_state()
        pre = f"bundled_k{k}_"
        out[pre + "draws_map"] = dm
        out[pre + "draws_ransac"] = dr
        out[pre + "used"] = np.array([used_m, used_r])
        out[pre + "N_before_after"] = np.array([n_before, r.N])
        out[pre + "x_map"] = x_map
        out[pre + "Pdiag_map"] = np.diag(P_map).copy()
        out[pre + "types"] = f_map["types"]
        out[pre + "init_uv"] = np.array([r.feature_init(i)[1][12:] for i in range(r.N)])
        out[pre + "has_h"] = f_s["has_h"]
        out[pre + "h"] = f_s["h"]
        out[pre + "S"] = f_s["S"]
        out[pre + "ic"] = f_s["ic"]
        out[pre + "z"] = f_s["z"]
        out[pre + "li"] = f_r["li"]
        out[pre + "hi"] = f_h["hi"]
        out[pre + "x"] = x
        if k < BUNDLED_FULL_P:
            out[pre + "P"] = P
        else:
            V = np.random.default_rng(1000 + k).standard_normal((P.shape[0], 4))
            out[pre + "Pdiag"] = np.diag(P).copy()
            out[pre + "PV"] = P @ V
        print(f"bundled frame {k}: N={r.N} ic={f_s['ic'].sum()} li={f_r['li'].sum()} hi={f_h['hi'].sum()} draws {used_m}+{used_r}")
    out["bundled_frames"] = np.array(BUNDLED_FRAMES)


def q1(out):
    for ci, (N, seed, frac) in enumerate(Q1_CASES):
        cam, x, P, z, ic = H.q1_consistent_state(N, seed=seed, outlier_frac=frac)
        r = R.ReferenceFilter()
        assert np.array_equal(r.camera9(), cam.as9())
        for i in range(N):
            r.add_feature(0, None, None, np.zeros(3), np.eye(3), z[i])
        r.set_state(x, P, prior=True)
        r.set_state(x, P, prior=False)
        r.predict_only()
        f0 = r.features()
        icm = ic & f0["has_h"]
        r.set_matches(z, icm)
        dr = R.make_draws(np.random.default_rng(100 + seed), 1000)
        r.set_draws(dr)
        r.ransac_hypotheses()
        used = r.draws_consumed()
        f1 = r.features()
        r.update_li()
        x_li, P_li = r.get_state()
        r.rescue_hi()
        f2 = r.features()
        r.update_hi()
        x_hi, P_hi = r.get_state()
        pre = f"q1_{ci}_"
        out[pre + "Nseedfrac"] = np.array([N, seed, frac])
        out[pre + "x_in"] = x
        out[pre + "P_in"] = P
        out[pre + "z"] = z
        out[pre + "ic"] = icm
        out[pre + "draws"] = dr
        out[pre + "used"] = np.array(used)
        out[pre + "h"] = f0["h"]
        out[pre + "S"] = f0["S"]
        out[pre + "li"] = f1["li"]
        out[pre + "hi"] = f2["hi"]
        out[pre + "x_li"] = x_li
        out[pre + "P_li"] = P_li
        out[pre + "x_hi"] = x_hi
        out[pre + "P_hi"] = P_hi
        out[pre + "h_rescue"] = f2["h"]
        print(f"q1 case {ci}: N={N} ic={icm.sum()} li={f1['li'].sum()} hi={f2['hi'].sum()} hypotheses run {used}")
    out["q1_cases"] = np.array(len(Q1_CASES))


def convert(out):
    N = 10
    cam, x, P, z, ic = H.q1_consistent_state(N, seed=21)
    # tighten rho of features 3 and 6 so that their linearity index drops under 0.1 (src/Map.cpp:146-147); only the first converts
    for i in (3, 6):
        s = 13 + 6 * i + 5
        P[s, :] *= 1e-3
        P[:, s] *= 1e-3
    r = R.ReferenceFilter()
    for i in range(N):
        r.add_feature(0, None, None, np.zeros(3), np.eye(3), z[i])
    r.set_state(x, P, prior=False)
    blank = np.full((240, 320), 90, np.uint8)
    dm = R.make_draws(np.random.default_rng(77), 200)
    r.set_draws(dm)
    r.map_management(blank, 5)
    xo, Po = r.get_state()
    f = r.features()
    out["convert_x_in"] = x
    out["convert_P_in"] = P
    out["convert_draws"] = dm
    out["convert_used"] = np.array(r.draws_consumed())
    out["convert_types"] = f["types"]
    out["convert_x"] = xo
    out["convert_P"] = Po
    # ... then a whole frame on the mixed map (one cartesian feature among inverse-depth ones: 3- and 6-wide state blocks): prediction,
    # h / H / S for both kinds (calculate_Hi_cartesian, src/Tracking.cpp:71-112), RANSAC and both updates with matches on the
    # inverse-depth features only (a matched cartesian feature makes the reference itself fail, SURVEY A.3 Q2)
    r.ekf_prediction()
    r.predict_only()
    f1 = r.features()
    icm = ic & f1["has_h"] & (f["types"] == 0)
    r.set_matches(z, icm)
    dr = R.make_draws(np.random.default_rng(78), 1000)
    r.set_draws(dr)
    r.ransac_hypotheses()
    used = r.draws_consumed()
    f2 = r.features()
    r.update_li()
    r.rescue_hi()
    f3 = r.features()
    r.update_hi()
    x2, P2 = r.get_state()
    out["convert_z"] = z
    out["convert_ic"] = icm
    out["convert_has_h"] = f1["has_h"]
    out["convert_h"] = f1["h"]
    out["convert_S"] = f1["S"]
    out["convert_H3"] = r.H_dense(3)
    out["convert_draws_ransac"] = dr
    out["convert_used_ransac"] = np.array(used)
    out["convert_li"] = f2["li"]
    out["convert_hi"] = f3["hi"]
    out["convert_x_frame"] = x2
    out["convert_P_frame"] = P2
    print("convert: types", f["types"], "n", xo.size, "draws", int(out["convert_used"]), "| frame: has_h", f1["has_h"].sum(), "ic", icm.sum(), "li", f2["li"].sum(), "hi",
          f3["hi"].sum(), "hyp", used)


if __name__ == "__main__":
    R.build()
    out = {}
    bundled(out)
    q1(out)
    convert(out)
    for path in golden_npz.save("ref_vectors", out):
        print("wrote", path, os.path.getsize(path) // 1024, "KiB")
