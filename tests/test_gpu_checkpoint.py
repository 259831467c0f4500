"""rslam_checkpoint_save / rslam_checkpoint_load: snapshots of whole filters that a slot of any handle continues from exactly.

Every comparison is bitwise (float64 as uint64, float32 as uint32).  The state of a slot is read back through the per-filter
download calls, which the snapshot path does not use."""
import importlib.util
import os
import re

import numpy as np
import pytest

from ransac_slam_b200 import synth
from tests import golden_npz

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "checkpoint_v1.bin")
STAGE = 256 << 20  # the library's staging buffer for host snapshots
NMAX = 110


_GEN = []


def _gen():
    """tests/golden/make_checkpoint_vectors.py as a module"""
    if not _GEN:
        spec = importlib.util.spec_from_file_location("make_checkpoint_vectors", os.path.join(ROOT, "tests", "golden", "make_checkpoint_vectors.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _GEN.append(mod)
    return _GEN[0]


_FRAMES = []


def _frames():
    if not _FRAMES:
        _FRAMES.append(golden_npz.load("pgm_frames_all")["frames"])
    return _FRAMES[0]


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else (a.view(np.uint32) if a.dtype == np.float32 else a)


def _assert_same(sa, sb, what):
    assert sa.keys() == sb.keys(), (what, sorted(sa), sorted(sb))
    for k in sa:
        a, b = np.asarray(sa[k]), np.asarray(sb[k])
        assert a.shape == b.shape, (what, k, a.shape, b.shape)
        assert np.array_equal(_bits(a), _bits(b)), (what, k)


def _snap(g, b):
    """everything the per-filter download calls show of slot b"""
    x, P = g.download_state(b=b)
    xp, _ = g.download_state(b=b, prior=True, want_P=False)
    Hc, Hf = g.H_sparse(b=b)
    s = dict(x=x, x_k_km1=xp, P=P, types=g.types(b=b), patches=g.download_patches(b=b), Hc=Hc, Hf=Hf, **g.features(b=b))
    N = len(s["types"])
    inits = [g.feature_init(i, b=b) for i in range(N)]
    s["patch41"] = np.array([p for p, _ in inits], dtype=np.uint8).reshape(N, 41, 41)
    s["pose14"] = np.array([q for _, q in inits]).reshape(N, 14)
    return s


def _member(seed, N, cartesian=()):
    """one filter's state and records (every field set; exactly symmetric P)"""
    scene, x, P = synth.random_spd_state(N, seed=seed)
    rng = np.random.default_rng(2000 + seed)
    types = np.zeros(N, np.int32)
    keep = np.ones(x.size, bool)
    for i in cartesian:
        types[i] = 1
        keep[13 + 6 * i + 3:13 + 6 * i + 6] = False
    x, P = x[keep], P[np.ix_(keep, keep)]
    return dict(cam9=scene.cam.as9(), std_z=scene.std_z, x=x, x_k_km1=x + rng.normal(0, 1e-3, x.size), P=np.asfortranarray((P + P.T) / 2), types=types,
                times_predicted=rng.integers(0, 20, N).astype(np.int32), times_measured=rng.integers(0, 20, N).astype(np.int32),
                flags=(rng.random((N, 4)) < 0.5).astype(np.uint8), h=rng.normal(160, 50, (N, 2)), Hc=rng.standard_normal((N, 2, 7)),
                Hf=rng.standard_normal((N, 2, 6)), z=rng.normal(160, 50, (N, 2)), templates=rng.integers(0, 256, (N, 13, 13)).astype(np.float64),
                patch41=rng.integers(0, 256, (N, 41, 41)).astype(np.uint8), r_wc=rng.standard_normal((N, 3)), R_wc=rng.standard_normal((N, 9)),
                uv=rng.uniform(20, 300, (N, 2)))


def _put(g, b, m, predict_S=False):
    G = _gen()
    G.load_into(g, b, m)
    if predict_S:  # S is only written by the prediction: run it, then put the chosen linearisation back
        g.L.rslam_predict_measurements(g.h)
        g.sync()
        g.upload_linearisation(m["h"], m["Hc"], m["Hf"], m["z"], m["flags"], b=b)


def _hetero():
    Ns = [20, 35, 50, 64, 80, 100, 27, 45]
    return [_member(100 + k, Ns[k % 8], cartesian=((1, 7) if k % 3 == 1 else ())) for k in range(16)]


def _handle(m, nmax=NMAX, batch=1, std_z=None):
    from ransac_slam_b200 import capi

    return capi.Filter(m["cam9"], nmax, batch=batch, std_z=m["std_z"] if std_z is None else std_z)


# ---- no GPU needed ------------------------------------------------------------------------------------------------------------------------------
def test_golden_file_matches_the_generator():
    from ransac_slam_b200 import capi

    G = _gen()
    buf = np.fromfile(GOLDEN, dtype=np.uint8)
    assert buf.size < (1 << 20)
    hdr, fl = capi.read_checkpoint(buf)
    ms = G.state()
    assert hdr["version"] == 1 and hdr["count"] == 2
    cam = ms[0]["cam9"]
    assert [hdr["camera"][k] for k in ("k1", "k2", "nRows", "nCols", "Cx", "Cy", "f", "dx", "dy")] == [float(v) if i not in (2, 3) else int(v) for i, v in enumerate(cam)]
    assert hdr["params"]["std_z"] == ms[0]["std_z"]
    for m, d in zip(ms, fl):
        _assert_same(d, G.expected(m), "golden filter")
    assert fl[1]["types"].tolist().count(1) == 1


def test_entry_points_are_declared_and_exported():
    import ctypes

    from ransac_slam_b200 import capi

    hdr = open(os.path.join(ROOT, "include", "rslam.h")).read()
    assert re.search(r"int rslam_checkpoint_bytes\(rslam_filter\* f, int b, int count, size_t\* bytes\);", hdr)
    assert re.search(r"int rslam_checkpoint_save\(rslam_filter\* f, int b, int count, void\* dst, size_t cap, size_t\* written\);", hdr)
    assert re.search(r"int rslam_checkpoint_load\(rslam_filter\* f, int b, const void\* src, size_t bytes, int\* count_out\);", hdr)
    if not os.path.exists(capi.LIB_PATH):
        pytest.skip("the CUDA library is not built")
    lib = ctypes.CDLL(capi.LIB_PATH)
    for s in ("rslam_checkpoint_bytes", "rslam_checkpoint_save", "rslam_checkpoint_load"):
        assert hasattr(lib, s), s


def test_read_checkpoint_refuses_foreign_bytes():
    from ransac_slam_b200 import capi

    buf = np.fromfile(GOLDEN, dtype=np.uint8)
    with pytest.raises(ValueError):
        capi.read_checkpoint(buf[:-16])
    bad = buf.copy()
    bad[0] ^= 1
    with pytest.raises(ValueError):
        capi.read_checkpoint(bad)


# ---- 6. the format pin on the GPU ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_golden_file_loads_and_saves_byte_for_byte():
    G = _gen()
    buf = np.fromfile(GOLDEN, dtype=np.uint8)
    g, ms = G.make_handle()
    assert g.load(buf) == 2
    for b, m in enumerate(ms):
        e = G.expected(m)
        s = _snap(g, b)
        for k in ("x", "x_k_km1", "P", "types", "patches", "patch41", "pose14", "h", "S", "z", "Hc", "Hf", "has_h", "ic", "li", "hi",
                  "times_predicted", "times_measured"):
            assert np.array_equal(_bits(np.asarray(s[k])), _bits(np.asarray(e[k]))), (b, k)
    again = g.save()
    assert again.size == buf.size and np.array_equal(again, buf)
    # and the same state built by the generator's uploads saves to the same bytes
    g2, _ = G.make_handle(batch=3, nmax=40)
    for b, m in enumerate(ms):
        G.load_into(g2, b + 1, m)
    assert np.array_equal(g2.save(1, 2), buf)


# ---- 1. round trip of a heterogeneous batch -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_round_trip_heterogeneous_batch():
    from ransac_slam_b200 import capi

    ms = _hetero()
    g = _handle(ms[0], batch=16)
    for b, m in enumerate(ms):
        _put(g, b, m, predict_S=True)
    ref = [_snap(g, b) for b in range(16)]
    assert any(np.abs(r["S"]).sum() > 0 for r in ref)
    buf = g.save()
    assert buf.size == g.checkpoint_bytes()
    # another handle: larger batch and max_features, loaded at slots 3..18; slots 0-2 and 19 hold other filters
    t = _handle(ms[0], nmax=130, batch=20)
    others = {b: _member(300 + b, 12 + b) for b in (0, 1, 2, 19)}
    for b, m in others.items():
        _put(t, b, m)
    before = {b: _snap(t, b) for b in others}
    assert t.load(buf, b=3) == 16
    for b in range(16):
        _assert_same(_snap(t, 3 + b), ref[b], f"loaded filter {b}")
        assert t.ransac_result(3 + b) == dict(status=0, hyp_run=0, best_support=0, n_hyp=0, num_ic=0, winner=0)
    for b in others:
        _assert_same(_snap(t, b), before[b], f"untouched slot {b}")
    # the numpy reader sees the same
    hdr, fl = capi.read_checkpoint(buf)
    assert hdr["count"] == 16
    for b in range(16):
        d = dict(fl[b])
        assert (d.pop("n"), d.pop("N")) == (ref[b]["x"].size, ref[b]["types"].size)
        _assert_same(d, ref[b], f"read_checkpoint filter {b}")
    # two saves of the same state are byte-for-byte equal, wherever the state sits
    assert np.array_equal(t.save(3, 16), buf)


# ---- 2. resume mid-run (into slots that held larger maps: a kernel that read past n / N would diverge) --------------------------------------------------------------------------------------------------------------------------
REPLAY_B, REPLAY_T, REPLAY_NMAX, REPLAY_MIN, NP, SAVE_AFTER = 8, 10, 80, 25, 60, 4


def _step_state(g, b):
    x, P = g.download_state(b=b)
    xp, _ = g.download_state(b=b, prior=True, want_P=False)
    return dict(x=x, x_k_km1=xp, P=P, types=g.types(b=b), **g.features(b=b))


@pytest.mark.gpu
def test_resume_mid_run_in_reversed_slots():
    from oracle import oracle_py as O
    from ransac_slam_b200 import capi

    frames = _frames()
    cam = synth.Camera()
    o0 = O.OracleFilter(cam.as9())
    o0.initialize_x_and_p()
    x0, P0 = o0.get_state()
    starts = [0, 11, 23, 35, 47, 59, 71, 83]
    g = capi.Filter(cam.as9(), REPLAY_NMAX, batch=REPLAY_B)
    for b in range(REPLAY_B):
        g.upload_state(x0, P0, feat_types=np.zeros(0, np.int32), b=b)
    g.set_patch_warp(True)
    rng = np.random.default_rng(17)
    r = None
    rev = list(range(REPLAY_B))[::-1]  # slot s of the resumed handle holds filter rev[s]
    for k in range(REPLAY_T):
        imgs = np.stack([frames[starts[b] + k] for b in range(REPLAY_B)])
        um = rng.random((REPLAY_B, 2 * NP))
        ur = rng.random((REPLAY_B, 1000))
        runs = [(g, imgs, um, ur, list(range(REPLAY_B)))] + ([(r, imgs[rev], um[rev], ur[rev], rev)] if r is not None else [])
        for h, im, u1, u2, _ in runs:
            for s in range(REPLAY_B):
                h.set_image(im[s], b=s)
            rc, status, info = h.map_management_batch(k + 1, REPLAY_MIN, u1, False)
            assert rc == 0, (k, status)
        if r is not None:
            for s in range(REPLAY_B):
                _assert_same(_step_state(r, s), _step_state(g, rev[s]), f"after map management {k}, filter {rev[s]}")
        for h, im, u1, u2, _ in runs:
            h.frame(im, u2)
        if r is not None:
            for s in range(REPLAY_B):
                _assert_same(_step_state(r, s), _step_state(g, rev[s]), f"after frame {k}, filter {rev[s]}")
                assert r.ransac_result(s) == g.ransac_result(rev[s]), (k, s)
        if k == SAVE_AFTER:
            r = capi.Filter(cam.as9(), REPLAY_NMAX, batch=REPLAY_B)
            r.set_patch_warp(True)
            for s in range(REPLAY_B):  # every slot first holds a larger map: P, x and records past the loaded n / N are not zero
                _put(r, s, _member(800 + s, REPLAY_NMAX - s))
            for s in range(REPLAY_B):
                assert r.load(g.save(rev[s], 1), b=s) == 1
    assert min(g.L.rslam_num_features(g.h, b) for b in range(REPLAY_B)) >= 10


# ---- 3. device memory ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_snapshot_equals_host_and_clones_a_filter():
    import torch

    ms = [_member(400 + k, 30 + 7 * k) for k in range(6)]
    g = _handle(ms[0], batch=6)
    for b, m in enumerate(ms):
        _put(g, b, m)
    host = g.save()
    dev = torch.empty(host.size + 64, dtype=torch.uint8, device="cuda:0")
    before = g.launches
    out = g.save(out=dev)
    assert g.launches - before == 2  # one chunk: the records and the covariance, one launch each
    assert out.numel() == host.size and np.array_equal(out.cpu().numpy(), host)
    # clone filter 2 into slot 5 on the device and run both on identical inputs
    one = torch.empty(g.checkpoint_bytes(2, 1), dtype=torch.uint8, device="cuda:0")
    g.save(2, 1, out=one)
    assert g.load(one, b=5) == 1
    _assert_same(_snap(g, 5), _snap(g, 2), "clone")
    frames = _frames()
    rng = np.random.default_rng(3)
    for k in range(3):
        imgs = np.stack([frames[10 * b + k] for b in range(6)])
        imgs[5] = imgs[2]
        u = rng.random((6, 1000))
        u[5] = u[2]
        g.frame(imgs, u)
        _assert_same(_snap(g, 5), _snap(g, 2), f"clone after frame {k}")
        assert g.ransac_result(5) == g.ransac_result(2)


# ---- 4. the chunked host path -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_chunked_host_path_large_map():
    """one filter at N = 2000: a 577 MB triangle in three chunks of the staging buffer"""
    import torch

    from ransac_slam_b200 import capi

    N = 2000
    cam = synth.scaled_camera(4)
    scene = synth.make_scene(N=N, seed=1234, cam=cam, margin=30, min_sep=18, assemble_P=False, motion_scale=0.25)
    dev = torch.device("cuda", 0)
    P0 = synth.assemble_P_torch(scene, dev)
    P0 = (P0 + P0.T) / 2
    n = scene.x0.size
    xd = torch.from_numpy(scene.x0.copy()).to(dev)
    g = capi.Filter(cam.as9(), N)
    g.upload_state_device(xd.data_ptr(), P0.data_ptr(), n, n, N)
    del P0
    nbytes = g.checkpoint_bytes()
    tri = 8 * n * (n + 1) // 2
    assert nbytes > tri > 2 * STAGE
    before = g.launches
    buf = g.save()
    chunks = g.launches - before - 1  # the records share the first chunk: one launch more than the chunks
    assert 3 <= chunks <= 4, chunks
    t = capi.Filter(cam.as9(), N + 50)
    assert t.load(buf) == 1
    xa, Pa = g.download_state()
    xb, Pb = t.download_state()
    assert np.array_equal(_bits(xa), _bits(xb))
    assert np.array_equal(_bits(Pa), _bits(Pb))
    del Pa, Pb
    assert np.array_equal(t.save(), buf)


@pytest.mark.gpu
def test_chunked_host_path_large_batch_and_launch_counts():
    """600 filters of 100 features (0.9 GB through the staging buffer); the launches follow the chunks, not the batch"""
    B = 600
    base = [_member(500 + k, 100) for k in range(8)]
    g = _handle(base[0], batch=B)
    rng = np.random.default_rng(9)
    for b in range(B):
        m = dict(base[b % 8])
        m["times_predicted"] = rng.integers(0, 50, 100).astype(np.int32)
        m["patch41"] = rng.integers(0, 256, (100, 41, 41)).astype(np.uint8)
        _put(g, b, m)
    nbytes = g.checkpoint_bytes()
    assert nbytes > 3 * STAGE
    before = g.launches
    buf = g.save()
    host_launches = g.launches - before
    assert 2 * (nbytes // STAGE) <= host_launches <= 2 * 2 * (nbytes // STAGE + 1), host_launches
    small = _handle(base[0], batch=16)
    for b in range(16):
        _put(small, b, base[b % 8])
    before = small.launches
    small.save()
    assert small.launches - before == 2
    t = _handle(base[0], batch=B)
    before = t.launches
    assert t.load(buf) == B
    assert t.launches - before == host_launches
    assert np.array_equal(t.save(), buf)
    for b in (0, 1, 299, 599):
        _assert_same(_snap(t, b), _snap(g, b), f"filter {b}")


# ---- loading over a larger map clears what lies past N --------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_load_over_a_larger_map_behaves_as_a_fresh_slot():
    small = _member(600, 10)
    big = _member(601, 60)
    src = _handle(small)
    _put(src, 0, small, predict_S=True)
    buf = src.save()
    dirty = _handle(small)
    _put(dirty, 0, big, predict_S=True)
    fresh = _handle(small)
    img = _frames()[0]
    for h in (dirty, fresh):
        h.load(buf)
        h.set_image(img)
        h.map_add_feature(np.array([150.0, 120.0]))
    _assert_same(_snap(dirty, 0), _snap(fresh, 0), "after a feature was added")
    assert dirty.N == 11


# ---- 5. refusals --------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_refusals_leave_the_handle_unchanged():
    from ransac_slam_b200 import capi
    from ransac_slam_b200.capi import _p

    ms = [_member(700, 20), _member(701, 30, cartesian=(4,))]
    src = _handle(ms[0], batch=2)
    for b, m in enumerate(ms):
        _put(src, b, m)
    buf = src.save()
    L = src.L

    def target(**kw):
        t = _handle(ms[0], batch=3, **kw)
        _put(t, 1, _member(702, 8))
        return t, [_snap(t, b) for b in range(3)]

    def refused(t, snaps, rc, code):
        assert rc == code, (rc, L.rslam_last_error())
        for b in range(3):
            _assert_same(_snap(t, b), snaps[b], f"slot {b} after a refusal")

    def load(t, data, b=0):
        data = np.ascontiguousarray(data, dtype=np.uint8)
        return L.rslam_checkpoint_load(t.h, b, _p(data), data.size, None)

    t, s = target()
    # asymmetric P: one upper entry changed
    bad = ms[1]["P"].copy(order="F")
    bad[2, 9] = np.nextafter(bad[2, 9], np.inf)
    src.upload_state(ms[1]["x"], bad, feat_types=ms[1]["types"], b=1)
    keep = _snap(src, 1)
    out = np.zeros(src.checkpoint_bytes(), np.uint8)
    assert L.rslam_checkpoint_save(src.h, 0, 2, _p(out), out.size, None) == -1
    assert "filter 1" in L.rslam_last_error().decode()
    _assert_same(_snap(src, 1), keep, "asymmetric filter after the refused save")
    assert L.rslam_checkpoint_save(src.h, 0, 1, _p(out), out.size, None) == 0  # filter 0 alone is fine
    # cap too small names the size
    assert L.rslam_checkpoint_save(src.h, 0, 1, _p(out), 100, None) == -1
    assert str(src.checkpoint_bytes(0, 1)) in L.rslam_last_error().decode()
    # N > max_features
    tc = _handle(ms[0], nmax=25, batch=3)
    _put(tc, 1, _member(702, 8))
    sc = [_snap(tc, b) for b in range(3)]
    refused(tc, sc, load(tc, buf), -3)
    # camera and params mismatch
    cam = list(ms[0]["cam9"])
    cam[4] += 1e-9
    tm = capi.Filter(cam, NMAX, batch=3, std_z=ms[0]["std_z"])
    refused(tm, [_snap(tm, b) for b in range(3)], load(tm, buf), -1)
    tp, sp = target(std_z=ms[0]["std_z"] * (1 + 1e-15))
    refused(tp, sp, load(tp, buf), -1)
    # bad magic, bad version, truncated, over-long, slots out of range
    b1 = buf.copy()
    b1[3] ^= 0x20
    refused(t, s, load(t, b1), -1)
    b2 = buf.copy()
    b2[8] = 2
    refused(t, s, load(t, b2), -1)
    refused(t, s, load(t, buf[:-8]), -1)
    refused(t, s, load(t, np.concatenate([buf, np.zeros(16, np.uint8)])), -1)
    refused(t, s, load(t, buf[:100]), -1)
    refused(t, s, load(t, buf, b=2), -1)
    refused(t, s, load(t, buf, b=-1), -1)
    # a table that lies about a filter's size
    b3 = buf.copy()
    b3[160 + 20] += 1
    refused(t, s, load(t, b3), -1)
    # and the good snapshot still loads
    assert t.load(buf, b=1) == 2
