"""More GPU parity cases through the C ABI: frozen golden vectors, edge cases the reference hits (no matches, zero-variance
patches, exhausted draws, cartesian features), batches, the hypothesis sweep, CUDA-graph replay, and size-independent
properties at the full N = 2000 size."""
import os

import numpy as np
import pytest

from oracle import np_oracle as NP
from oracle import oracle_py as O
from ransac_slam_b200 import synth, sweep
from tests import helpers as H

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.mark.parametrize("tag", ["ref", "noq1"])
def test_golden_vectors(tag):
    g = np.load(os.path.join(GOLD, "oracle_vectors.npz"))
    N, seed, quirks = int(g[f"{tag}_N"]), int(g[f"{tag}_seed"]), int(g[f"{tag}_quirks"])
    scene, x, P = synth.random_spd_state(N, seed=seed)
    seq = synth.make_sequence(scene, T=1, seed=seed + 5, t0=3)
    f = H.gpu_from(scene, x, P, quirks=H.quirks_o2g(quirks))
    f.set_image(seq.images[0])
    f.search_ic_matches()
    ft = f.features()
    assert (ft["ic"] == g[f"{tag}_ic"]).all() and (ft["z"][ft["ic"]] == g[f"{tag}_z"][ft["ic"]]).all()
    np.testing.assert_allclose(ft["S"][ft["has_h"]], g[f"{tag}_S"][ft["has_h"]], rtol=1e-9)
    res = f.ransac_hypotheses(seq.u01[0])
    assert [res["status"], res["hyp_run"], res["best_support"], res["n_hyp"], res["num_ic"]] == list(g[f"{tag}_info"])
    assert (f.features()["li"] == g[f"{tag}_li"]).all()
    f.update_li()
    xg, Pg = f.download_state()
    H.assert_x_close(xg, g[f"{tag}_x_li"])
    H.assert_P_close(Pg, g[f"{tag}_P_li"])
    f.rescue_hi()
    assert (f.features()["hi"] == g[f"{tag}_hi"]).all()
    f.update_hi()
    xg, Pg = f.download_state()
    H.assert_x_close(xg, g[f"{tag}_x_hi"])
    H.assert_P_close(Pg, g[f"{tag}_P_hi"])


def test_edge_no_matches_is_a_noop():
    scene, x, P = synth.random_spd_state(10, seed=61)
    f = H.gpu_from(scene, x, P)
    f.set_image(np.zeros((scene.cam.nRows, scene.cam.nCols), np.uint8))  # zero-variance candidates -> NaN scores -> unmatched (Q10)
    f.search_ic_matches()
    assert not f.features()["ic"].any()
    res = f.ransac_hypotheses(np.random.default_rng(0).random(100))
    assert res["status"] == 1 and res["num_ic"] == 0 and res["winner"] == -1  # Q9
    f.update_li()
    f.rescue_hi()
    f.update_hi()
    xk, Pk = f.download_state()
    assert np.array_equal(xk, x) and np.array_equal(Pk, P)


def test_edge_uniform_draws_exhausted():
    scene, x, P = synth.random_spd_state(10, seed=61)
    seq = synth.make_sequence(scene, T=1, seed=66, t0=3)
    o = H.oracle_from(scene, x, P)
    f = H.gpu_from(scene, x, P)
    o.search_ic_matches(seq.images[0])
    f.set_image(seq.images[0])
    f.search_ic_matches()
    rc, info = o.ransac_hypotheses(seq.u01[0][:5])
    res = f.ransac_hypotheses(seq.u01[0][:5])
    assert rc == res["status"] == 3 and info["hyp_run"] == res["hyp_run"] == 5


def test_mixed_cartesian_features_predict_and_ub_guard():
    from ransac_slam_b200 import capi

    scene, x, P = synth.random_spd_state(12, seed=71)
    # convert features 2, 5, 9 to cartesian: state shrinks by 3 each
    types = np.zeros(12, int)
    types[[2, 5, 9]] = 1
    keep, xs = list(range(13)), []
    for i in range(12):
        o6 = 13 + 6 * i
        if types[i] == 0:
            keep += list(range(o6, o6 + 6))
        else:
            keep += [o6, o6 + 1, o6 + 2]
    xm = x[keep].copy()
    Pm = np.asfortranarray(P[np.ix_(keep, keep)])
    pos = 13
    for i in range(12):
        if types[i] == 1:
            xm[pos:pos + 3] = scene.landmarks[i] + 0.001 * np.random.default_rng(i).standard_normal(3)
            pos += 3
        else:
            pos += 6
    o = H.oracle_from(scene, xm, Pm, feat_types=types)
    f = H.gpu_from(scene, xm, Pm, feat_types=types)
    o.search_ic_matches(None)
    f.search_ic_matches()
    fo, fg = o.features(), f.features()
    assert (fo["has_h"] == fg["has_h"]).all() and fo["has_h"].sum() >= 10
    v = fo["has_h"]
    np.testing.assert_allclose(fg["h"][v], fo["h"][v], atol=1e-9, rtol=0)
    np.testing.assert_allclose(fg["S"][v], fo["S"][v], rtol=1e-9, atol=1e-12)
    Hc, Hf = f.H_sparse()
    offs = 13 + np.concatenate([[0], np.cumsum(np.where(types == 0, 6, 3))])[:-1]
    for i in np.flatnonzero(v):
        Hd = o.H_dense(i)
        fs = 6 if types[i] == 0 else 3
        np.testing.assert_allclose(Hc[i], Hd[:, :7], rtol=1e-9, atol=1e-11)
        np.testing.assert_allclose(Hf[i][:, :fs], Hd[:, offs[i]:offs[i] + fs], rtol=1e-9, atol=1e-11)
    # a matched cartesian feature: the reference's support scoring is undefined (Q2) -> explicit error, never a silent answer
    z = fo["h"].round()
    ic = np.ones(12, np.uint8)
    o.set_matches(z, ic)
    f.set_matches(z, ic)
    rc, _ = o.ransac_hypotheses(np.full(10, 0.5))
    assert rc == 2
    with pytest.raises(capi.RslamError):
        f.ransac_hypotheses(np.full(10, 0.5))
    # the joint update itself handles mixed maps: inject inlier flags through a cartesian-free RANSAC is not possible, so use hi path
    ic2 = (types == 0).astype(np.uint8)
    o.set_matches(z, ic2)
    f.set_matches(z, ic2)
    u = np.random.default_rng(5).random(1000)
    o.ransac_hypotheses(u)
    f.ransac_hypotheses(u)
    o.update_li(); f.update_li()
    o.rescue_hi(); f.rescue_hi()
    assert (o.features()["hi"] == f.features()["hi"]).all()
    o.update_hi(); f.update_hi()
    xo, Po = o.get_state()
    xg, Pg = f.download_state()
    H.assert_x_close(xg, xo)
    H.assert_P_close(Pg, Po)


def test_batch_matches_single_and_graph_matches_stream():
    scene = synth.make_scene(N=30, seed=81)
    seq = synth.make_sequence(scene, T=3, seed=82)
    ref = H.gpu_from(scene, scene.x0, scene.P0, prior=False)
    ref.set_graph(False)
    bat = H.gpu_from(scene, scene.x0, scene.P0, prior=False, batch=3)
    for k in range(3):
        ref.frame(seq.images[k][None], seq.u01[k][None])
        bat.frame(np.repeat(seq.images[k][None], 3, 0), np.repeat(seq.u01[k][None], 3, 0))
    gra = H.gpu_from(scene, scene.x0, scene.P0, prior=False)  # single filter again, frame replayed as a CUDA graph
    for k in range(3):
        gra.frame(seq.images[k][None], seq.u01[k][None])
    xr, Pr = ref.download_state()
    xg, Pg = gra.download_state()
    # same kernels, same order (the graph captures the side-stream fork / join of W beside S + Cholesky as parallel branches): bitwise
    assert np.array_equal(xr, xg) and np.array_equal(Pr, Pg)
    x0, P0 = bat.download_state(b=0)
    for b in range(3):
        xb, Pb = bat.download_state(b=b)
        assert np.array_equal(x0, xb) and np.array_equal(P0, Pb), b  # members of a batch: bitwise
        # a batch forms S = H W from the stored W, a single filter straight from P (different summation order): 1e-9 bar
        H.assert_x_close(xb, xr, what=f"batch member {b} vs single")
        H.assert_P_close(Pb, Pr, what=f"batch member {b} vs single")
        assert (bat.features(b)["hi"] == ref.features()["hi"]).all()


def test_prefetched_inputs_give_the_same_frames_as_inline_copies():
    """rslam_prefetch_inputs (copy stream + second staging set) only changes WHEN the host inputs are copied: trajectories must be bitwise
    equal to the inline-copy path, also when a staged set is dropped because the next frame is handed other buffers."""
    import torch

    scene = synth.make_scene(N=30, seed=83)
    T = 5
    seq = synth.make_sequence(scene, T=T, seed=84)
    inline = H.gpu_from(scene, scene.x0, scene.P0, prior=False)
    for k in range(T):
        inline.frame(seq.images[k][None], seq.u01[k][None])
    xi, Pi = inline.download_state()
    rows, cols = seq.images.shape[1:]
    himg = torch.from_numpy(seq.images).pin_memory()
    hu = torch.from_numpy(seq.u01).pin_memory()
    nu = seq.u01.shape[1]

    def args(k):
        return (himg.data_ptr() + k * rows * cols, rows, cols, cols), (hu.data_ptr() + k * nu * 8, nu)

    pf = H.gpu_from(scene, scene.x0, scene.P0, prior=False)
    for k in range(T):
        pf.frame(*args(k))  # frame 0 copies inline, frames 1.. consume the staged set
        if k + 1 < T:
            pf.prefetch(*args(k + 1))
        if k == 2:
            pf.prefetch(*args(0))  # staged, then overwritten by the right one: the last prefetch wins
            pf.prefetch(*args(k + 1))
    xp, Pp = pf.download_state()
    assert np.array_equal(xi, xp) and np.array_equal(Pi, Pp)
    # a staged set that does not match the next frame's buffers is dropped, not used
    dr = H.gpu_from(scene, scene.x0, scene.P0, prior=False)
    for k in range(T):
        dr.prefetch(*args((k + 2) % T))
        dr.frame(*args(k))
    xd, Pd = dr.download_state()
    assert np.array_equal(xi, xd) and np.array_equal(Pi, Pd)
    # arguments that cannot be staged
    du = torch.zeros(nu, dtype=torch.float64, device="cuda")
    with pytest.raises(Exception):
        pf.prefetch(args(0)[0], (du.data_ptr(), nu))  # device-resident inputs need no staging


@pytest.mark.parametrize("q1", [True, False])
def test_support_sweep_against_numpy(q1):
    scene, x, P = synth.random_spd_state(40, seed=91)
    seq = synth.make_sequence(scene, T=1, seed=96, t0=3)
    quirks = 0x7 if q1 else 0x6
    cam = scene.cam.as9()
    types = np.zeros(scene.N, int)
    rng = np.random.default_rng(4)
    hyp = rng.integers(0, 30, 500).astype(np.int32)
    results = []
    for dedupe in (True, False):
        f = H.gpu_from(scene, x, P, quirks=quirks, dedupe=dedupe)
        f.set_image(seq.images[0])
        f.search_ic_matches()
        ft = f.features()
        nic = int(ft["ic"].sum())
        assert nic >= 30
        key, mask, pairs = f.support_sweep(hyp)
        results.append((key, mask[:nic].copy(), pairs))
        assert pairs == (len(np.unique(hyp)) if dedupe else len(hyp)) * nic
        # sharded: max of the shard keys == global key
        keys = [f.support_sweep(hyp, *sweep.shard_range(len(hyp), 4, r), want_mask=False)[0] for r in range(4)]
        assert max(keys) == key
        # sharded by match index instead (how the deduplicated sweep scales over GPUs)
        keys_m = [f.support_sweep(hyp, want_mask=False, match_begin=sweep.shard_range(nic, 3, r)[0], match_end=sweep.shard_range(nic, 3, r)[1])[0] for r in range(3)]
        assert max(keys_m) == key
    assert results[0][0] == results[1][0] and (results[0][1] == results[1][1]).all()
    # numpy restatement of every distinct hypothesis
    o = H.oracle_from(scene, x, P)
    o.search_ic_matches(seq.images[0])
    fo = o.features()
    ic = np.flatnonzero(fo["ic"])
    sup = {}
    for t in np.unique(hyp):
        p = ic[t]
        sup[t] = NP.hypothesis_support(cam, x, P, types, o.H_dense(p), fo["h"][p], fo["z"][p], fo["z"], fo["ic"], q1=q1)
    supports = np.array([sup[t][0] for t in hyp])
    exp_key = sweep.local_key(supports, 0)
    assert results[0][0] == exp_key, (sweep.decode_key(results[0][0]), sweep.decode_key(exp_key))
    s, hid = sweep.decode_key(exp_key)
    if s > 0:
        assert (results[0][1] == sup[hyp[hid]][1]).all()


def test_full_size_properties_N2000():
    """N = 2000 (state dim 12013, P 1.15 GB): size-independent properties of one frame + numpy check of the li/hi update algebra
    on a sub-block (the dense oracle would need hours here)."""
    import torch

    from ransac_slam_b200 import capi

    N = 2000
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
    seq = synth.make_sequence(scene, T=1, seed=1235, n_u01=2048)
    dev = torch.device("cuda", 0)
    P0 = synth.assemble_P_torch(scene, dev)
    n = scene.x0.size
    f = capi.Filter(cam.as9(), N, quirks=0x6, std_a=0.007 * 0.25, std_alpha=0.007 * 0.25)  # Q1 off: a real li set
    x0 = torch.from_numpy(scene.x0).to(dev)
    f.upload_state_device(x0.data_ptr(), P0.data_ptr(), n, n, N)
    f.upload_patches(scene.templates.astype(np.float64))
    tr0 = float(torch.trace(P0))
    f.begin_frame()
    f.ekf_prediction()
    f.set_image(seq.images[0])
    f.search_ic_matches()
    res = f.ransac_hypotheses(seq.u01[0])
    ft = f.features()
    assert ft["ic"].sum() > 1500 and res["best_support"] > 800
    xp, Pp = f.download_state(prior=True)  # x_k_km1 and P_k_km1 (in-place covariance, before any update)
    Hc, Hf = f.H_sparse()
    f.update_li()
    xl, Pl = f.download_state()
    assert np.array_equal(Pl, Pl.T)
    assert abs(np.linalg.norm(xl[3:7]) - 1) < 1e-12
    assert np.trace(Pl) < np.trace(Pp)
    d = np.diag(Pp) - np.diag(Pl)
    assert d.min() > -1e-9 * np.abs(np.diag(Pp)).max()  # variances never grow (outside the Jnorm rows)
    # numpy / LAPACK restatement of the same update from the downloaded prior (dense reference formula, BLAS threaded)
    li = np.flatnonzero(ft["li"])
    k = 2 * li.size
    Hd = np.zeros((k, n))
    for t, i in enumerate(li):
        Hd[2 * t:2 * t + 2, :7] = Hc[i]
        Hd[2 * t:2 * t + 2, 13 + 6 * i:19 + 6 * i] = Hf[i]
    z = ft["z"][li].reshape(-1)
    h = ft["h"][li].reshape(-1)
    xn, Pn = NP.ekf_update(xp, Pp, Hd, z, h)
    H.assert_x_close(xl, xn, rtol=1e-9)
    H.assert_P_close(Pl, Pn, rtol=1e-9)
    f.rescue_hi()
    f.update_hi()
    xh, Ph = f.download_state()
    assert np.array_equal(Ph, Ph.T) and np.trace(Ph) <= np.trace(Pl) and np.isfinite(Ph).all()
    assert tr0 > 0


def test_patch_warp_matches_oracle_remap():
    """Tracking::pred_patch_fc on the device (homography warp + cv::remap-compatible sampling) against the oracle, whose remap is
    pinned bit-exactly to cv2 (tests/golden/cv_fixtures.npz).  Then a search with the warped patches on both sides."""
    N = 40
    scene, x, P = synth.random_spd_state(N, seed=111)
    rng = np.random.default_rng(5)
    # smooth-ish 41x41 appearance so that the warped patch still correlates with the image content
    init = rng.integers(0, 256, (N, 41, 41)).astype(np.uint8)
    o = O.OracleFilter(scene.cam.as9(), std_z=scene.std_z, quirks=O.Q_ALL, sparse=False, fast_corr=True, warp_patches=True)
    for i in range(N):
        o.add_feature(0, init[i], None, scene.x0[:3], np.eye(3), scene.uv0[i])
    o.set_state(x, P, prior=True)
    g = H.gpu_from(scene, x, P)
    g.upload_feature_init(init, np.tile(scene.x0[:3], (N, 1)), np.tile(np.eye(3).reshape(1, 9), (N, 1)), scene.uv0)
    g.set_patch_warp(True)
    o.search_ic_matches(None)
    g.search_ic_matches()
    pg = g.download_patches()
    fo = o.features()
    assert fo["has_h"].sum() >= N - 2
    same, npix, neq, worst = 0, 0, 0, 0.0
    for i in np.flatnonzero(fo["has_h"]):
        po = o.patch_matching(i)
        assert po.std() > 0
        d = np.abs(pg[i].astype(np.float64) - po)
        # identical sampling except where a map coordinate sits within rounding noise (1e-13 px) of a 1/32-px quantisation boundary
        assert (d == 0).mean() > 0.99 and d.max() < 12.0, (i, (d == 0).mean(), d.max())
        same += int((d == 0).all())
        npix += d.size
        neq += int((d == 0).sum())
        worst = max(worst, float(d.max()))
    stats = f"patch warp vs oracle: {same}/{int(fo['has_h'].sum())} patches identical, {neq}/{npix} pixels identical, max |d| = {worst}"
    print(stats)
    assert neq >= npix - 2, stats  # bit-identical pixels (a flip needs a coordinate within ~1e-13 px of a quantisation boundary)
    # build an image that contains the oracle-predicted appearance at a pasted location and search on both sides
    img = synth.background(scene.cam).copy()
    for i in np.flatnonzero(fo["has_h"]):
        cx, cy = np.rint(fo["h"][i]).astype(int)
        if 7 <= cx < scene.cam.nCols - 7 and 7 <= cy < scene.cam.nRows - 7:
            img[cy - 6:cy + 7, cx - 6:cx + 7] = np.clip(np.rint(o.patch_matching(i)), 0, 255).astype(np.uint8)
    o.search_ic_matches(img)
    g.set_image(img)
    g.search_ic_matches()
    f2o, f2g = o.features(), g.features()
    assert f2o["ic"].sum() >= N // 2
    assert (f2o["ic"] == f2g["ic"]).all() and (f2o["z"][f2o["ic"]] == f2g["z"][f2g["ic"]]).all()


def test_upload_linearisation_reproduces_the_update_and_stage_entry_points():
    """rslam_upload_linearisation (what the host ExtendKF::update uses when it is handed caller-built H, z, h) and the two halves of
    search_IC_matches as separate entry points (Tracking::calculate_derivatives / matching)."""
    import ctypes as C

    scene, x, P = synth.random_spd_state(40, seed=131)
    seq = synth.make_sequence(scene, T=1, seed=136, t0=3)
    a = H.gpu_from(scene, x, P, quirks=0x6)
    a.set_image(seq.images[0])
    a.search_ic_matches()
    a.ransac_hypotheses(seq.u01[0])
    fa = a.features()
    Hc, Hf = a.H_sparse()
    assert fa["li"].sum() >= 5
    a.update_li()
    xa, Pa = a.download_state()
    # second handle: prediction and matching as separate calls, then the linearisation + flags of the first injected instead of RANSAC
    b = H.gpu_from(scene, x, P, quirks=0x6)
    b.set_image(seq.images[0])
    L = b.L
    assert L.rslam_predict_measurements(b.h) == 0 and L.rslam_match(b.h) == 0
    fb = b.features()
    assert (fb["ic"] == fa["ic"]).all() and np.array_equal(fb["z"][fb["ic"]], fa["z"][fa["ic"]]) and np.array_equal(fb["h"], fa["h"])
    flags = np.stack([fa["has_h"], fa["ic"], fa["li"], np.zeros_like(fa["li"])], axis=1).astype(np.uint8)
    arrs = [np.ascontiguousarray(v, dtype=np.float64) for v in (fa["h"], Hc, Hf, fa["z"])]
    rc = L.rslam_upload_linearisation(b.h, 0, *[v.ctypes.data_as(C.c_void_p) for v in arrs], np.ascontiguousarray(flags).ctypes.data_as(C.c_void_p))
    assert rc == 0
    b.update_li()
    xb, Pb = b.download_state()
    assert np.array_equal(xa, xb) and np.array_equal(Pa, Pb)
