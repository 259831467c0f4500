"""rslam_map_management_batch: Map::map_management for every filter of a batch in one fixed launch sequence.

Every member must come out bitwise equal to a batch-1 handle that holds the same state, records, flags, image and uniforms and
runs rslam_map_management (the per-filter path, itself pinned to the oracle by test_gpu_map.py), except where the batched call
deliberately differs: a member whose delete pass is undefined in the reference is left untouched, and bad arguments are refused
before any work."""
import os
import re

import numpy as np
import pytest

from oracle import oracle_py as O
from ransac_slam_b200 import synth
from tests import golden_npz
from tests import helpers as H

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NMAX = 110
NP = 60  # uniform pairs per member (>= 50)

_FRAMES = []


def _frames():
    if not _FRAMES:
        _FRAMES.append(golden_npz.load("pgm_frames_all")["frames"])
    return _FRAMES[0]


def _member(seed, N, deletes=(), convert=None, measured=0, cartesian=(), hidden=False, img=None):
    """state, records and inputs of one filter: `deletes` get counters that the delete pass removes, feature `convert` a rho variance
    that makes it pass the linearity test, the first `measured` features the li flag; `hidden` turns every feature away from the
    camera, so that no feature blocks the sampling box"""
    scene, x, P = synth.random_spd_state(N, seed=seed)
    rng = np.random.default_rng(1000 + seed)
    types = np.zeros(N, np.int32)
    keep = np.ones(x.size, bool)
    for i in cartesian:  # a cartesian feature keeps the first 3 of its 6 rows
        types[i] = 1
        keep[13 + 6 * i + 3:13 + 6 * i + 6] = False
    if hidden:
        for i in range(N):
            if types[i] == 0:
                x[13 + 6 * i + 3] = np.pi
    if convert is not None:
        ip = 13 + 6 * convert
        s = 1e-3 / np.sqrt(P[ip + 5, ip + 5])
        P[ip + 5, :] *= s
        P[:, ip + 5] *= s
    x, P = x[keep], np.asfortranarray(P[np.ix_(keep, keep)])
    tp = np.full(N, 10, np.int32)
    tm = np.full(N, 9, np.int32)
    tm[list(deletes)] = 1
    flags = np.zeros((N, 4), np.uint8)
    flags[:, 0] = rng.random(N) < 0.7
    flags[:, 1] = rng.random(N) < 0.5
    flags[:measured, 2] = 1
    rec = dict(h=rng.normal(160, 50, (N, 2)), Hc=rng.standard_normal((N, 2, 7)), Hf=rng.standard_normal((N, 2, 6)), z=rng.normal(160, 50, (N, 2)),
               flags=flags, tp=tp, tm=tm, patches41=rng.integers(0, 256, (N, 41, 41)).astype(np.uint8), r_wc=rng.standard_normal((N, 3)),
               R_wc=rng.standard_normal((N, 9)), uv=rng.uniform(20, 300, (N, 2)), templates=rng.uniform(0, 255, (N, 13, 13)))
    frames = _frames()
    return dict(cam=scene.cam, std_z=scene.std_z, x=x, P=P, types=types, rec=rec, img=frames[seed % len(frames)] if img is None else img,
                u01=rng.random(2 * NP))


def _load(g, b, m):
    g.upload_state(m["x"], m["P"], feat_types=m["types"], b=b, prior=False)
    r = m["rec"]
    g.set_counters(r["tp"], r["tm"], b=b)
    g.upload_linearisation(r["h"], r["Hc"], r["Hf"], r["z"], r["flags"], b=b)
    g.upload_patches(r["templates"], b=b)
    g.upload_feature_init(r["patches41"], r["r_wc"], r["R_wc"], r["uv"], b=b)
    g.set_image(m["img"], b=b)


def _filter(members, nmax=NMAX):
    from ransac_slam_b200 import capi

    m0 = members[0]
    g = capi.Filter(m0["cam"].as9(), nmax, batch=len(members), std_z=m0["std_z"])
    for b, m in enumerate(members):
        _load(g, b, m)
    return g


def _snap(g, b):
    x, P = g.download_state(b=b)
    s = dict(x=x, P=P, types=g.types(b=b), patches=g.download_patches(b=b), **g.features(b=b))
    N = len(s["types"])
    inits = [g.feature_init(i, b=b) for i in range(N)]
    s["patch41"] = np.array([p for p, _ in inits]).reshape(N, 41, 41)
    s["pose14"] = np.array([q for _, q in inits]).reshape(N, 14)
    return s


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else (a.view(np.uint32) if a.dtype == np.float32 else a)


def _assert_same(sa, sb, what):
    for k in sa:
        assert sa[k].shape == sb[k].shape, (what, k, sa[k].shape, sb[k].shape)
        assert np.array_equal(_bits(sa[k]), _bits(sb[k])), (what, k)


def _single_call(g, step, min_features, u01, reference_indexing):
    """rslam_map_management on a batch-1 handle: (rc, info) for every rc, capacity included"""
    from ransac_slam_b200.capi import _p

    u = np.ascontiguousarray(u01, dtype=np.float64)
    info = np.zeros(4, np.int32)
    rc = g.L.rslam_map_management(g.h, 0, int(step), int(min_features), int(reference_indexing), _p(u), u.size // 2, _p(info))
    assert rc in (0, -3, -4), g.L.rslam_last_error()
    return rc, list(info)


def _singles(members, step, min_features, reference_indexing, nmax=NMAX, before=None):
    """each member on its own batch-1 handle through rslam_map_management; before(g) runs first"""
    out = []
    for m in members:
        g = _filter([m], nmax)
        if before:
            before(g, m)
        out.append(_single_call(g, step, min_features, m["u01"], reference_indexing) + (_snap(g, 0),))
        g.close()
    return out


def _batch_u01(members):
    return np.stack([m["u01"] for m in members])


def _hetero_members():
    ms = []
    for k in range(16):
        N = [20, 35, 50, 64, 80, 100, 27, 45][k % 8]
        dels = [(), (3,), (2, 7, 11), (1, 4)][k % 4]
        ms.append(_member(seed=40 + k, N=N, deletes=dels, convert=(5 if k % 3 == 0 else None), measured=[0, 5, 11, 20][k % 4] if N < 100 else 20,
                          cartesian=((9,) if k % 5 == 1 and len(dels) <= 1 else ()), hidden=(k % 2 == 0)))
    return ms


@pytest.mark.gpu
@pytest.mark.parametrize("reference_indexing", [True, False])
def test_batch_equals_singles_bitwise(reference_indexing):
    ms = _hetero_members()
    ref = _singles(ms, 3, 12, reference_indexing)
    g = _filter(ms)
    rc, status, info = g.map_management_batch(3, 12, _batch_u01(ms), reference_indexing)
    for b in range(len(ms)):
        rcs, infos, ss = ref[b]
        assert status[b] == rcs and list(info[b]) == infos, (b, status[b], rcs, list(info[b]), infos)
        _assert_same(_snap(g, b), ss, f"member {b}")
    assert rc == next((s for s in status if s != 0), 0)
    assert (info[:, 0] > 0).any() and (info[:, 1] >= 0).any() and (info[:, 2] > 0).any(), info


@pytest.mark.gpu
def test_edge_members_reference_ub_and_capacity():
    nmax = 40
    ub = _member(seed=7, N=6, deletes=(1, 5))  # run-ahead index past the end at the second deletion
    cap = _member(seed=8, N=37, measured=0, hidden=True)  # every accepted corner fits until max_features
    ok1 = _member(seed=9, N=30, deletes=(2,), convert=4, measured=15, hidden=True)
    ok2 = _member(seed=10, N=25, measured=25)
    ms = [ub, cap, ok1, ok2]
    ref = _singles(ms, 2, 20, True, nmax=nmax)
    g = _filter(ms, nmax)
    before = _snap(g, 0)
    rc, status, info = g.map_management_batch(2, 20, _batch_u01(ms), True)
    assert list(status) == [-4, -3, 0, 0] and rc == -4, status
    assert list(info[0]) == [1, -1, 0, 0], info[0]
    _assert_same(_snap(g, 0), before, "reference-UB member")
    assert ref[0][0] == -4
    for b in (1, 2, 3):
        rcs, infos, ss = ref[b]
        assert status[b] == rcs and list(info[b]) == infos, (b, status[b], rcs, list(info[b]), infos)
        _assert_same(_snap(g, b), ss, f"member {b}")
    assert g.L.rslam_num_features(g.h, 1) == nmax


@pytest.mark.gpu
def test_mixed_with_per_filter_calls():
    ms = [_member(seed=21 + k, N=30 + 5 * k, deletes=((3,) if k != 1 else ()), convert=(2 if k == 2 else None), measured=4, hidden=True) for k in range(3)]
    ref = _singles(ms, 1, 10, True, before=lambda g, m: g.map_delete_feature(6))
    g = _filter(ms)
    for b in range(3):
        g.map_delete_feature(6, b=b)
    rc, status, info = g.map_management_batch(1, 10, _batch_u01(ms), True)
    for b in range(3):
        rcs, infos, ss = ref[b]
        assert status[b] == rcs and list(info[b]) == infos
        _assert_same(_snap(g, b), ss, f"member {b}")


@pytest.mark.gpu
def test_fixed_launch_sequence():
    """the same launches at B = 1 and B = 16, with no edit at all and with deletions, conversions and additions"""
    quiet1 = [_member(seed=31, N=20)]
    busy1 = [_member(seed=31, N=20, deletes=(3,), convert=5, hidden=True)]
    quiet16 = [_member(seed=60 + k, N=20 + 5 * k) for k in range(16)]
    busy16 = _hetero_members()
    counts = []
    for ms, edits in ((quiet1, False), (busy1, True), (quiet16, False), (busy16, True)):
        g = _filter(ms)
        before = g.launches
        rc, status, info = g.map_management_batch(1, 12 if edits else 0, _batch_u01(ms), True)
        counts.append(g.launches - before)
        if edits:
            assert (info[:, 0] > 0).any() and (info[:, 1] >= 0).any() and (info[:, 2] > 0).any(), info
        else:
            assert rc == 0 and (info[:, 0] == 0).all() and (info[:, 1] == -1).all() and (info[:, 2] == 0).all(), info
    assert len(set(counts)) == 1, counts


@pytest.mark.gpu
def test_large_map_equals_single():
    """B = 1, N = 2000 (P = 1.15 GB): a deletion, a conversion and an addition in one call"""
    import torch

    from ransac_slam_b200 import capi

    N = 2000
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
    dev = torch.device("cuda", 0)
    P0 = synth.assemble_P_torch(scene, dev)
    n = scene.x0.size
    x0 = scene.x0.copy()
    x0[13 + 3::6] = np.pi  # no feature blocks the sampling box
    ip = 13 + 6 * 700
    s = 1e-3 / torch.sqrt(P0[ip + 5, ip + 5])
    P0[ip + 5, :] *= s
    P0[:, ip + 5] *= s
    tp = np.full(N, 10, np.int32)
    tm = np.full(N, 9, np.int32)
    tm[300] = 1
    img = np.tile(_frames()[0], (4, 4))
    u01 = np.random.default_rng(5).random(2 * NP)
    xd = torch.from_numpy(x0).to(dev)
    out = []
    for batched in (False, True):
        g = capi.Filter(cam.as9(), N + 1)
        g.upload_state_device(xd.data_ptr(), P0.data_ptr(), n, n, N)
        g.set_counters(tp, tm)
        g.set_image(img)
        if batched:
            rc, status, info = g.map_management_batch(1, 1, u01[None], True)
            res = (rc, list(info[0]))
        else:
            res = _single_call(g, 1, 1, u01, True)
        x, P = g.download_state()
        out.append((res, x, P, g.types()))
        g.close()
        del P
    (ra, xa, Pa, ta), (rb, xb, Pb, tb) = out
    assert ra == rb and ra[1][0] == 1 and ra[1][1] >= 0 and ra[1][2] == 1, (ra, rb)
    assert np.array_equal(ta, tb)
    assert np.array_equal(_bits(xa), _bits(xb)) and np.array_equal(_bits(Pa), _bits(Pb))
    assert np.array_equal(Pb, Pb.T)


@pytest.mark.gpu
def test_argument_checks_leave_the_handle_untouched():
    ms = [_member(seed=51, N=20, deletes=(2,), convert=3), _member(seed=52, N=25, deletes=(1,))]
    g = _filter(ms)
    before = [_snap(g, b) for b in range(2)]
    L = g.L
    st = np.zeros(2, np.int32)
    u = _batch_u01(ms)
    from ransac_slam_b200.capi import _p

    assert L.rslam_map_management_batch(g.h, 1, 10, 1, _p(u[:, :98].copy()), 49, _p(st), None) == -1
    assert L.rslam_map_management_batch(g.h, 1, 10, 1, None, NP, _p(st), None) == -1
    assert L.rslam_map_management_batch(g.h, 1, 10, 1, _p(u), NP, None, None) == -1
    from ransac_slam_b200 import capi

    g4 = capi.Filter(ms[0]["cam"].as9(), NMAX, batch=2, std_z=ms[0]["std_z"])  # no image bound to filter 1
    for b in range(2):
        g4.upload_state(ms[b]["x"], ms[b]["P"], feat_types=ms[b]["types"], b=b, prior=False)
    g4.set_image(ms[0]["img"], b=0)
    b4 = [_snap(g4, b) for b in range(2)]
    assert L.rslam_map_management_batch(g4.h, 1, 10, 1, _p(u), NP, _p(st), None) == -1
    for b in range(2):
        _assert_same(_snap(g, b), before[b], f"member {b}")
        _assert_same(_snap(g4, b), b4[b], f"member {b} without image")


def test_symbol_is_exported_and_declared():
    """no GPU needed"""
    import ctypes

    from ransac_slam_b200 import capi

    hdr = open(os.path.join(ROOT, "include", "rslam.h")).read()
    assert re.search(r"int rslam_map_management_batch\(rslam_filter\* f, int step, int min_features, int reference_indexing, const double\* u01, int n_pairs, int\* status,\s*int\* info4\);", hdr)
    if not os.path.exists(capi.LIB_PATH):
        pytest.skip("the CUDA library is not built")
    assert hasattr(ctypes.CDLL(capi.LIB_PATH), "rslam_map_management_batch")


# ---- the whole TrackRunning loop (consistent deletion: the run-ahead index is covered above) --------------------------------------------------------------------------------------------------
REPLAY_B, REPLAY_T, REPLAY_NMAX, REPLAY_MIN = 8, 10, 80, 25


def _pair_reference_step(g2, step, um, reference_indexing=False):
    """rslam_map_management's order with the per-filter primitives on a batch-2 handle holding one filter twice"""
    nd, conv, init, att, rcs = [], [], [], [], []
    for bb in range(2):
        rc, d = g2.map_delete_features(reference_indexing, b=bb)
        assert rc == 0
        nd.append(d)
    meas = [int((lambda f: (f["li"] | f["hi"]).sum())(g2.features(b=bb))) for bb in range(2)]
    g2.begin_frame()
    for bb in range(2):
        conv.append(g2.map_inversedepth_to_cartesian(b=bb))
        target = REPLAY_MIN if meas[bb] == 0 else (REPLAY_MIN - meas[bb] if meas[bb] < REPLAY_MIN else 0)
        ni, at = g2.map_initialize_features(step, target, um, b=bb) if target > 0 else (0, 0)
        init.append(ni)
        att.append(at)
    assert nd[0] == nd[1] and conv[0] == conv[1] and init[0] == init[1] and att[0] == att[1]
    return [nd[0], conv[0], init[0], att[0]]


@pytest.mark.gpu
def test_replay_whole_loop_against_pairs_and_oracle():
    from ransac_slam_b200 import capi

    frames = _frames()
    cam = synth.Camera()
    o0 = O.OracleFilter(cam.as9())
    o0.initialize_x_and_p()
    x0, P0 = o0.get_state()
    starts = [0, 11, 23, 35, 47, 59, 71, 83]
    g = capi.Filter(cam.as9(), REPLAY_NMAX, batch=REPLAY_B)
    pairs = []
    for b in range(REPLAY_B):
        g.upload_state(x0, P0, feat_types=np.zeros(0, np.int32), b=b)
        g2 = capi.Filter(cam.as9(), REPLAY_NMAX, batch=2)
        for bb in range(2):
            g2.upload_state(x0, P0, feat_types=np.zeros(0, np.int32), b=bb)
        g2.set_patch_warp(True)
        pairs.append(g2)
    g.set_patch_warp(True)
    oracles = {}
    for b in (0, 5):
        o = O.OracleFilter(cam.as9())
        o.initialize_x_and_p()
        o.set_options(O.Q_ALL, sparse=False, fast_corr=True, warp_patches=True)
        oracles[b] = o
    rng = np.random.default_rng(17)
    for k in range(REPLAY_T):
        imgs = np.stack([frames[starts[b] + k] for b in range(REPLAY_B)])
        um = rng.random((REPLAY_B, 2 * NP))
        ur = rng.random((REPLAY_B, 1000))
        for b in range(REPLAY_B):
            g.set_image(imgs[b], b=b)
        rc, status, info = g.map_management_batch(k + 1, REPLAY_MIN, um, False)
        assert rc == 0, (k, status)
        for b in range(REPLAY_B):
            g2 = pairs[b]
            for bb in range(2):
                g2.set_image(imgs[b], b=bb)
            ref = _pair_reference_step(g2, k + 1, um[b])
            assert list(info[b]) == ref, (k, b, list(info[b]), ref)
            assert np.array_equal(g.types(b=b), g2.types(b=0))
            xa, Pa = g.download_state(b=b)
            xb, Pb = g2.download_state(b=0)
            assert np.array_equal(_bits(xa), _bits(xb)) and np.array_equal(_bits(Pa), _bits(Pb)), (k, b)
            if b in oracles:
                rco, io = oracles[b].map_management(imgs[b], k + 1, REPLAY_MIN, um[b], False)
                assert (rco, [io["deleted"], io["converted"], io["initialised"], io["attempts"]]) == (0, ref), (k, b, io)
                xo, Po = oracles[b].get_state()
                H.assert_x_close(xa, xo, what=f"x after map management, frame {k}, filter {b}")
                H.assert_P_close(Pa, Po, what=f"P after map management, frame {k}, filter {b}")
        g.frame(imgs, ur)
        for b in range(REPLAY_B):
            g2 = pairs[b]
            g2.frame(np.stack([imgs[b], imgs[b]]), np.stack([ur[b], ur[b]]))
            fa, fb = g.features(b=b), g2.features(b=0)
            for key in ("ic", "li", "hi"):
                assert np.array_equal(fa[key], fb[key]), (k, b, key)
            assert g.ransac_result(b) == g2.ransac_result(0), (k, b)
            xa, Pa = g.download_state(b=b)
            xb, Pb = g2.download_state(b=0)
            assert np.array_equal(_bits(xa), _bits(xb)) and np.array_equal(_bits(Pa), _bits(Pb)), (k, b)
            if b in oracles:
                oracles[b].frame(imgs[b], ur[b])
                fo = oracles[b].features()
                for key in ("ic", "li", "hi"):
                    assert (fo[key] == fa[key]).all(), (k, b, key)
                xo, Po = oracles[b].get_state()
                H.assert_x_close(xa, xo, what=f"x after frame {k}, filter {b}")
                H.assert_P_close(Pa, Po, what=f"P after frame {k}, filter {b}")
    assert min(g.L.rslam_num_features(g.h, b) for b in range(REPLAY_B)) >= 10
