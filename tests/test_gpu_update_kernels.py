"""The joint EKF update -- W = P H^T, S = H W + I, Cholesky, triangular solve, P -= V V^T with the fused state correction, quaternion
normalisation -- against a float64 numpy reference, at chosen innovation sizes, map sizes, batches and tuning switches.

In a whole frame RANSAC decides k = 2m, so frame tests cannot be steered onto the edges of the update's kernels.  Here the state, the
covariance, the linearisation and the inlier flags are uploaded directly (rslam_upload_state / rslam_upload_linearisation) and
rslam_update_li / rslam_update_hi run exactly the update.  Every case names the kernel route it exists for; `route()` restates the
selection rules of run_update (ransac_slam_b200/csrc/rslam_api.cu) and each GPU case checks the per-launch profile against it, so a
later change to the dispatch cannot silently move a case off its target.  Template variants share a profile name; for those the
rule in `route()` is the evidence.

The reference is oracle/np_oracle.py::ekf_update on the dense H.  The tests that check the reference itself (two formulations agree;
the data would expose a lost measurement) need no GPU."""
import functools

import numpy as np
import pytest
import scipy.linalg

from oracle import np_oracle as NP
from ransac_slam_b200 import synth
from tests import helpers as H

CAM9 = synth.Camera().as9()
Q_ALL, Q4 = 0x7, 0x2
SWITCHES = ("RSLAM_TRSM_OB", "RSLAM_CHOL_OUTER_SMALL", "RSLAM_CHOL2")  # the ones that steer run_update


def cdiv(a, b):
    return -(-a // b)


# ---- inputs ---------------------------------------------------------------------------------------------------------------------
def feature_layout(types):
    sizes = np.where(types == 0, 6, 3)
    offs = 13 + np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(int)
    return offs, sizes, 13 + int(sizes.sum())


@functools.lru_cache(maxsize=6)
def make_map(N, cart=(), seed=0):
    """Feature types (cartesian at the positions `cart`), x and P of a map of N features.  Returns (types, x, P); cached, read only."""
    rng = np.random.default_rng([N, seed, 11])
    types = np.zeros(N, np.int32)
    types[list(cart)] = 1
    offs, sizes, n = feature_layout(types)
    x = np.zeros(n)
    sd = np.zeros(n)
    x[0:3] = np.array([0.12, -0.05, 0.3]) + rng.normal(0, 0.01, 3)
    q = np.array([0.97, 0.06, -0.2, 0.04]) + rng.normal(0, 0.01, 4)
    x[3:7] = q / np.linalg.norm(q) * (1 + 1e-3 * rng.choice([-1.0, 1.0]))  # 1e-3 off unit norm: the normalisation has work to do
    x[7:10] = rng.normal(0, 0.01, 3)
    x[10:13] = rng.normal(0, 0.005, 3)
    sd[0:3], sd[3:7], sd[7:10], sd[10:13] = 0.004, 0.001, 0.01, 0.003
    for i in range(N):
        o = offs[i]
        if types[i] == 0:
            rho = 1.0 / rng.uniform(2.0, 15.0)
            x[o:o + 3] = x[0:3] + rng.normal(0, 0.05, 3)
            x[o + 3] = rng.uniform(-0.5, 0.5)
            x[o + 4] = rng.uniform(-0.4, 0.4)
            x[o + 5] = rho
            sd[o:o + 3], sd[o + 3:o + 5], sd[o + 5] = 0.002, 0.001, 0.3 * rho
        else:
            x[o:o + 3] = x[0:3] + np.array([rng.uniform(-2, 2), rng.uniform(-1.5, 1.5), rng.uniform(3, 10)])
            sd[o:o + 3] = 0.03
    # P = D (a U U^T / r + diag(d)) D: every entry non-zero, SPD, O(n^2 r) to build
    r, a = 6, 0.1
    U = rng.standard_normal((n, r)) * np.sqrt(a / r)
    C = U @ U.T
    C[np.diag_indices(n)] += rng.uniform(0.5, 1.5, n)
    P = np.asfortranarray(C * sd[:, None] * sd[None, :])
    P = np.asfortranarray(0.5 * (P + P.T))
    for v in (x, P, types):
        v.flags.writeable = False
    return types, x, P


@functools.lru_cache(maxsize=6)
def make_linearisation(N, cart=(), seed=0, lin_seed=0):
    """Hc (N, 2, 7), Hf (N, 2, 6), h, z (N, 2) for the map make_map(N, cart, seed).  H entries O(1), each row scaled so that its
    H P H^T diagonal entry is 10..100 px^2 (the downdate V V^T is then comparable to P); innovations z - h of O(1) px.  The unused
    columns 3..5 of a cartesian feature's Hf are large finite values: the device must ignore them (the dense H never sees them)."""
    types, x, P = make_map(N, cart, seed)
    offs, sizes, n = feature_layout(types)
    rng = np.random.default_rng([N, seed, lin_seed, 12])
    Hc = rng.standard_normal((N, 2, 7))
    Hf = rng.standard_normal((N, 2, 6))
    for i in range(N):
        fs = sizes[i]
        idx = np.r_[0:7, offs[i]:offs[i] + fs]
        Ps = P[np.ix_(idx, idx)]
        for row in range(2):
            g = np.r_[Hc[i, row], Hf[i, row, :fs]]
            s = np.sqrt(rng.uniform(10.0, 100.0) / (g @ Ps @ g))
            Hc[i, row] *= s
            Hf[i, row, :fs] *= s
        if fs == 3:
            Hf[i, :, 3:] = rng.choice([-1.0, 1.0], (2, 3)) * 1e9
    h = np.column_stack([rng.uniform(5, 315, N), rng.uniform(5, 235, N)])
    z = h + rng.standard_normal((N, 2))
    for v in (Hc, Hf, h, z):
        v.flags.writeable = False
    return Hc, Hf, h, z


def inlier_set(N, k, seed=0):
    """k / 2 inliers at random positions; features 0 and N - 1 are always among them (N - 1 alone when k = 2)."""
    assert k % 2 == 0 and 0 <= k <= 2 * N
    m = k // 2
    inl = np.zeros(N, bool)
    if m == 0:
        return inl
    inl[N - 1] = True
    if m >= 2:
        inl[0] = True
        rng = np.random.default_rng([N, k, seed, 13])
        inl[1 + rng.choice(N - 2, m - 2, replace=False)] = True
    assert inl.sum() == m
    return inl


def dense_H(types, lin, inl):
    """Stacked dense H (k x n), z and h of the inliers in feature order (the order of the device's gather)."""
    Hc, Hf, h, z = lin
    offs, sizes, n = feature_layout(types)
    idx = np.flatnonzero(inl)
    Hd = np.zeros((2 * idx.size, n))
    for t, i in enumerate(idx):
        Hd[2 * t:2 * t + 2, :7] = Hc[i]
        Hd[2 * t:2 * t + 2, offs[i]:offs[i] + sizes[i]] = Hf[i, :, :sizes[i]]
    return Hd, z[idx].reshape(-1), h[idx].reshape(-1)


def reference(types, x, P, lin, inl, q4=True):
    Hd, z, h = dense_H(types, lin, inl)
    return NP.ekf_update(x, P, Hd, z, h, q4_int_exponent=q4)


def reference_cholesky(types, x, P, lin, inl, q4=True):
    """The same update through a Cholesky factorisation of S instead of np_oracle's explicit inverse."""
    Hd, z, h = dense_H(types, lin, inl)
    W = P @ Hd.T
    c = scipy.linalg.cho_factor(Hd @ W + np.eye(z.size), lower=True)
    xkk = x + W @ scipy.linalg.cho_solve(c, z - h)
    Pt = P - W @ scipy.linalg.cho_solve(c, W.T)
    return NP.normalise_quaternion(xkk, 0.5 * Pt + 0.5 * Pt.T, q4)


@functools.lru_cache(maxsize=4)
def fresh_reference(N, cart, seed, lin_seed, k, q4):
    """reference() of one update of the map make_map(N, cart, seed) as generated (cached, read only)."""
    types, x, P = make_map(N, cart, seed)
    xr, Pr = reference(types, x, P, make_linearisation(N, cart, seed, lin_seed), inlier_set(N, k, lin_seed), q4)
    xr.flags.writeable = Pr.flags.writeable = False
    return xr, Pr


# ---- the route run_update takes -------------------------------------------------------------------------------------------------
def route(N, n, B, trsm_ob=16, chol_outer_small=True, chol2=True):
    """Launches per profile name and the template variants run_update chooses for a handle whose largest uploaded map has N features
    and whose largest state has n entries (B filters; switches as rslam_create read them).  Restates rslam_api.cu:236-342."""
    kmax, nsteps = 2 * N, cdiv(2 * N, 64)
    launches = {"k_upd_gather": 1, "k_upd_W": 1, "k_upd_S": 1, "k_chol_trinv": 1, "k_upd_jnorm": 1}
    v = {"jnorm": "wide" if n >= 4096 else "narrow"}
    if kmax <= 256:
        v["S"] = "direct" if B == 1 else "batched"
        v["chol_small"] = (212, 2) if B > 1 and chol2 and kmax <= 200 and B >= 2 * 148 else (260, 1)
        v["syrk_kpad"] = cdiv(kmax, 32) * 32
        launches.update({"k_chol_small": 1, "k_trsm_small": 1, "k_syrk_rows": 1})
        return launches, v
    launches["k_chol_panel"] = nsteps
    v["chol_outer"] = []
    for s in range(nsteps):
        o = 64 * (s + 1)
        if kmax <= o:
            break
        if (s + 1) % 4 == 0:
            ts = cdiv(kmax - o, 64)
            v["chol_outer"].append((64, 64) if chol_outer_small and ts * (ts + 1) // 2 * B <= 8 * 444 else (128, 64))
    if v["chol_outer"]:
        launches["k_gemm_dmma/chol_outer"] = len(v["chol_outer"])
    ob = trsm_ob if trsm_ob > 0 else nsteps
    nouter = cdiv(nsteps, ob)
    launches["k_trsm_ll"] = nouter
    v["trsm_ll"] = (48, 2) if cdiv(n + 1, 48) * B >= 200 else (32, 2)
    v["trsm_outer_at"] = [64 * ob * (J + 1) for J in range(nouter) if kmax > 64 * ob * (J + 1)]
    if v["trsm_outer_at"]:
        launches["k_gemm_dmma/trsm_outer"] = len(v["trsm_outer_at"])
    tm = cdiv(n + 1, 128)
    v["syrk_P"] = (128, 64) if tm * (tm + 1) * B >= 192 else (64, 64)
    launches["k_gemm_dmma/syrk_P"] = 1
    return launches, v


def test_route_restates_the_dispatch_for_the_table():
    """The rule above puts every map of the case table on the route the table names (no GPU needed)."""
    _, v = route(128, 781, 1)
    assert v == {"jnorm": "narrow", "S": "direct", "chol_small": (260, 1), "syrk_kpad": 256}
    assert route(128, 781, 2)[1]["S"] == "batched"
    l, v = route(129, 787, 1)
    assert v["chol_outer"] == [(64, 64)] and l["k_chol_panel"] == 5 and v["trsm_ll"] == (32, 2) and v["syrk_P"] == (64, 64)
    assert "k_gemm_dmma/trsm_outer" not in l
    l, v = route(600, 3610, 1)
    assert v["chol_outer"] == [(64, 64)] * 4 and v["trsm_outer_at"] == [1024] and v["syrk_P"] == (128, 64) and v["trsm_ll"] == (32, 2)
    assert route(600, 3610, 1, chol_outer_small=False)[1]["chol_outer"] == [(128, 64)] * 4
    assert route(600, 3610, 1, trsm_ob=3)[1]["trsm_outer_at"] == [192, 384, 576, 768, 960, 1152]
    assert route(600, 3610, 1, trsm_ob=0)[0]["k_trsm_ll"] == 1
    assert route(680, 4093, 1)[1]["jnorm"] == "narrow" and route(681, 4096, 1)[1]["jnorm"] == "wide"
    l, v = route(800, 4813, 2)
    assert v["trsm_ll"] == (48, 2) and v["jnorm"] == "wide" and route(800, 4813, 1)[1]["trsm_ll"] == (32, 2)


# ---- checks of the reference itself (no GPU) -----------------------------------------------------------------------------------
# one case per map size of the GPU cases: (N, cartesian positions, k)
SIZES = [(128, (), 256), (129, (), 258), (600, (599,), 1200), (680, (), 1360), (681, (0,), 1362), (650, (), 1026), (800, (), 1600)]


@pytest.mark.parametrize("N,cart,k", SIZES, ids=[f"N{s[0]}-k{s[2]}" for s in SIZES])
def test_reference_is_well_conditioned_and_sensitive(N, cart, k):
    """The reference built with an explicit inverse and with a Cholesky solve agrees to 1e-12 (the data are well conditioned, so the
    1e-9 bar measures the device, not the reference); dropping the last inlier pair moves x or P by more than 1e-6 relative (1000x
    the bar: a lost measurement or a lost 64-column block cannot hide)."""
    types, x, P = make_map(N, cart)
    lin = make_linearisation(N, cart)
    inl = inlier_set(N, k)
    xa, Pa = reference(types, x, P, lin, inl)
    xb, Pb = reference_cholesky(types, x, P, lin, inl)
    H.assert_x_close(xa, xb, rtol=1e-12)
    H.assert_P_close(Pa, Pb, rtol=1e-12)
    short = inl.copy()
    short[np.flatnonzero(inl)[-1]] = False
    xs, Ps = reference(types, x, P, lin, short)
    moved = max(np.abs(Ps - Pa).max() / np.abs(Pa).max(), np.abs(xs - xa).max() / np.abs(xa).max())
    assert moved > 1e-6, moved
    # the masked Hf entries of cartesian features are large: had they entered the reference, nothing would agree
    assert all(np.abs(lin[1][i, :, 3:]).min() >= 1e9 for i in cart)


# ---- the device -------------------------------------------------------------------------------------------------------------------
class Handle:
    """A capi.Filter of B filters created under the given tuning switches, plus a host mirror of what its update should produce."""

    def __init__(self, monkeypatch, max_features, batch=1, quirks=Q_ALL, env=None):
        from ransac_slam_b200 import capi

        env = env or {}
        for name in SWITCHES:
            monkeypatch.delenv(name, raising=False)
        for name, val in env.items():
            monkeypatch.setenv(name, str(val))
        self.f = capi.Filter(CAM9, max_features, batch=batch, quirks=quirks)  # rslam_create reads the switches
        self.B, self.q4 = batch, bool(quirks & Q4)
        self.sw = dict(trsm_ob=int(env.get("RSLAM_TRSM_OB", 16)), chol_outer_small=int(env.get("RSLAM_CHOL_OUTER_SMALL", 1)) != 0,
                       chol2=int(env.get("RSLAM_CHOL2", 1)) != 0)
        self.maps = [None] * batch  # (N, cart, seed, n) per member
        self.mirror = [None] * batch  # (types, x_km1, x_kk, P) per member: what the reference says the device holds
        self.held = [None] * batch  # (x_kk, P) per member: what the device last returned (or was given)

    def upload(self, b, N, cart=(), seed=0, prior=True):
        """Upload map make_map(N, cart, seed) as x_k_km1 (prior) or x_k_k, with its P."""
        types, x, P = make_map(N, cart, seed)
        self.f.upload_state(x, P, feat_types=types, b=b, prior=prior)
        self.maps[b] = (N, cart, seed, x.size)
        self.mirror[b] = (types, x if prior else None, None if prior else x, P)
        self.held[b] = (None if prior else x, P)

    def linearise(self, b, k, which, lin_seed=0):
        N, cart, seed, _ = self.maps[b]
        lin = make_linearisation(N, cart, seed, lin_seed)
        inl = inlier_set(N, k, lin_seed)
        flags = np.zeros((N, 4), np.uint8)
        flags[:, 0] = 1
        flags[:, 1] = 1
        flags[:, 2 + which] = inl
        self.f.upload_linearisation(lin[2], lin[0], lin[1], lin[3], flags, b=b)
        return lin, inl, lin_seed

    def route(self):
        up = [m for m in self.maps if m is not None]
        return route(max(m[0] for m in up), max(m[3] for m in up), self.B, **self.sw)

    def update(self, which, lins, profile=True):
        """Run update_li (which = 0) / update_hi (1) on every member with the linearisations `lins` ({b: linearise(b, ...)}), check the
        launches against route() and every member against the reference.  Returns the downloaded states."""
        f = self.f
        if profile:
            f.profile(True)
            f.profile_read()
        (f.update_hi if which else f.update_li)()
        if profile:
            launches = {name: cnt for name, (cnt, _) in f.profile_read().items()}
            f.profile(False)
            expect, _ = self.route()
            assert launches == expect
        out = {}
        for b, (lin, inl, lin_seed) in lins.items():
            types, x_km1, x_kk, P = self.mirror[b]
            N, cart, seed, _ = self.maps[b]
            _, x_map, P_map = make_map(N, cart, seed)
            base = x_kk if which else x_km1
            xg, Pg = f.download_state(b=b)
            what = f"member {b}, k = {2 * int(inl.sum())}"
            assert np.array_equal(Pg, Pg.T), what
            if not inl.any():  # no measurements: x_k_k = the base state, P untouched, bit for bit (src/ExtendKF.cpp:635-638)
                assert np.array_equal(xg, self.held[b][0] if which else x_km1), what
                assert np.array_equal(Pg, self.held[b][1]), what
                xr, Pr = base, P
            else:
                if base is x_map and P is P_map:  # straight from the upload: several cases share this reference
                    xr, Pr = fresh_reference(N, cart, seed, lin_seed, 2 * int(inl.sum()), self.q4)
                else:
                    xr, Pr = reference(types, base, P, lin, inl, self.q4)
                H.assert_x_close(xg, xr, what="x " + what)
                H.assert_P_close(Pg, Pr, what="P " + what)
            self.mirror[b] = (types, x_km1, xr, Pr)  # the next reference starts from the reference's result
            self.held[b] = (xg, Pg)
            out[b] = (xg, Pg)
        return out

    def close(self):
        self.f.close()


@pytest.fixture
def handles():
    made = []
    yield made
    for h in made:
        h.close()


def single(monkeypatch, handles, N, k, cart=(), which=0, quirks=Q_ALL, env=None, max_features=None):
    """One filter: upload the map, one update with k inliers, check it.  Returns (handle, downloaded x, P)."""
    h = Handle(monkeypatch, max_features or N, quirks=quirks, env=env)
    handles.append(h)
    h.upload(0, N, cart, prior=which == 0)
    lin = h.linearise(0, k, which)
    xg, Pg = h.update(which, {0: lin})[0]
    return h, xg, Pg


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 64, 66, 200, 254, 256])
def test_small_path_top_single_filter(monkeypatch, handles, k):
    """kmax = 256, the top of the single-filter latency path: k_upd_S_direct + k_upd_W, k_chol_small<260, 1>, k_trsm_small,
    k_syrk_rows with K padded to 256.  Profiling keeps one stream; the same update without it (k_upd_W on the side stream) must
    give the same bits."""
    h, xg, Pg = single(monkeypatch, handles, 128, k)
    assert h.route()[1] == {"jnorm": "narrow", "S": "direct", "chol_small": (260, 1), "syrk_kpad": 256}
    h.upload(0, 128)
    lin = h.linearise(0, k, 0)
    xf, Pf = h.update(0, {0: lin}, profile=False)[0]
    assert np.array_equal(xf, xg) and np.array_equal(Pf, Pg)


@pytest.mark.gpu
def test_small_path_batch_with_different_and_empty_members(monkeypatch, handles):
    """The batched small path (k_upd_S): two members of 128 features with k = (256, 2), then (0, 130) on the updated covariances."""
    h = Handle(monkeypatch, 128, batch=2)
    handles.append(h)
    h.upload(0, 128, seed=0)
    h.upload(1, 128, seed=1)
    assert h.route()[1]["S"] == "batched"
    h.update(0, {0: h.linearise(0, 256, 0), 1: h.linearise(1, 2, 0)})
    h.update(0, {0: h.linearise(0, 0, 0, lin_seed=1), 1: h.linearise(1, 130, 0, lin_seed=1)})


@pytest.mark.gpu
@pytest.mark.parametrize("k", [0, 2, 64, 256, 258])
def test_large_path_smallest_case(monkeypatch, handles, k):
    """N = 129, the smallest large-path handle: five panels, one K = 256 chol_outer, then a 2-wide last panel; k_trsm_ll<32, 2> in
    one outer block; k_gemm_dmma<64, 64> syrk_P; k = 0 on the large path."""
    h, _, _ = single(monkeypatch, handles, 129, k)
    l, v = h.route()
    assert l["k_chol_panel"] == 5 and v["chol_outer"] == [(64, 64)] and v["trsm_ll"] == (32, 2) and v["syrk_P"] == (64, 64)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 254, 256, 258, 510, 512, 514, 1022, 1024, 1026, 1200])
def test_large_path_block_boundaries_odd_rows(monkeypatch, handles, k):
    """N = 600 with one cartesian feature, last (n + 1 = 3611 odd): k around the 64-wide panel, the 256-wide Cholesky outer block and
    the 1024-wide TRSM outer block; k_gemm_dmma<128, 64> syrk_P over an odd number of rows."""
    h, _, _ = single(monkeypatch, handles, 600, k, cart=(599,))
    _, v = h.route()
    assert (h.f.n + 1) % 2 == 1 and v["syrk_P"] == (128, 64) and v["trsm_outer_at"] == [1024]


@pytest.mark.gpu
@pytest.mark.parametrize("q4", [True, False], ids=["q4", "no-q4"])
@pytest.mark.parametrize("N,cart,k", [(680, (), 1360), (681, (0,), 1362)], ids=["n4093", "n4096"])
def test_jnorm_wide_switch_edge(monkeypatch, handles, N, cart, k, q4):
    """n = 4093 (k_upd_jnorm, one CTA) vs n = 4096 (k_upd_jnorm_wide at its first size, 16 CTAs; cartesian feature first), with the
    quaternion Jacobian's reference exponent (Q4) and the analytic one."""
    h, _, _ = single(monkeypatch, handles, N, k, cart=cart, quirks=Q_ALL if q4 else Q_ALL & ~Q4)
    assert h.route()[1]["jnorm"] == ("wide" if N == 681 else "narrow")


@pytest.mark.gpu
def test_large_path_batch_of_different_maps(monkeypatch, handles):
    """B = 2 with maps of 800 and 650 features (n = 4813 / 3913): k_trsm_ll<48, 2>, grids sized for the larger member, the wide
    jnorm on the smaller one; k = (1600, 0), then (1026, 2) on the updated covariances."""
    h = Handle(monkeypatch, 800, batch=2)
    handles.append(h)
    h.upload(0, 800)
    h.upload(1, 650)
    _, v = h.route()
    assert v["trsm_ll"] == (48, 2) and v["jnorm"] == "wide" and v["trsm_outer_at"] == [1024]
    h.update(0, {0: h.linearise(0, 1600, 0), 1: h.linearise(1, 0, 0)})
    h.update(0, {0: h.linearise(0, 1026, 0, lin_seed=1), 1: h.linearise(1, 2, 0, lin_seed=1)})


@pytest.mark.gpu
def test_leading_dimensions_larger_than_the_map(monkeypatch, handles):
    """N = 129 on a handle sized for 600 features: ldp / ldw / lds are those of the larger capacity, not the tight values."""
    single(monkeypatch, handles, 129, 258, max_features=600)


@pytest.mark.gpu
@pytest.mark.parametrize("N,cart,k", [(129, (), 258), (600, (599,), 1026)], ids=["N129", "N600"])
def test_hi_update(monkeypatch, handles, N, cart, k):
    """The high-innovation update: base state x_k_k, which = 1 in the syrk_P epilogue."""
    single(monkeypatch, handles, N, k, cart=cart, which=1)


@pytest.mark.gpu
@pytest.mark.parametrize("N,cart,k_li,k_hi", [(128, (), 200, 64), (600, (599,), 1200, 514)], ids=["small", "large"])
def test_li_then_hi_on_one_handle(monkeypatch, handles, N, cart, k_li, k_hi):
    """A low-innovation update, a second linearisation uploaded, then the high-innovation update from the first one's x_k_k and P
    (k_syrk_rows and k_gemm_dmma epilogues with the x_k_k base)."""
    h = Handle(monkeypatch, N)
    handles.append(h)
    h.upload(0, N, cart)
    h.update(0, {0: h.linearise(0, k_li, 0)})
    h.update(1, {0: h.linearise(0, k_hi, 1, lin_seed=1)})


@pytest.mark.gpu
def test_smaller_updates_after_larger_ones(monkeypatch, handles):
    """One handle (600 features of capacity): W / S / Linv keep stale columns beyond the current k, which every kernel must mask.
    k = 1200, 130, 0 on the 600-feature map; a 100-feature map (small path, k = 200); the 600-feature map again with k = 1026."""
    h = Handle(monkeypatch, 600)
    handles.append(h)
    h.upload(0, 600, (599,))
    h.update(0, {0: h.linearise(0, 1200, 0)})
    h.update(0, {0: h.linearise(0, 130, 0, lin_seed=1)})
    h.update(0, {0: h.linearise(0, 0, 0, lin_seed=2)})
    h.upload(0, 100)
    assert "k_syrk_rows" in h.route()[0]
    h.update(0, {0: h.linearise(0, 200, 0)})
    h.upload(0, 600, (599,))
    assert "k_gemm_dmma/syrk_P" in h.route()[0]
    h.update(0, {0: h.linearise(0, 1026, 0)})


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1026, 1200])
@pytest.mark.parametrize("ob", [0, 1, 3, 16])
def test_trsm_outer_block_width(monkeypatch, handles, ob, k):
    """RSLAM_TRSM_OB regroups the triangular solve (0: one left-looking launch; 3: 192-wide outer blocks, which do not line up with the
    Cholesky's 256): every width at the bar."""
    single(monkeypatch, handles, 600, k, cart=(599,), env={"RSLAM_TRSM_OB": ob})


@pytest.mark.gpu
@pytest.mark.parametrize("N,cart,k", [(600, (599,), 1200), (129, (), 258)], ids=["N600", "N129"])
def test_chol_outer_tile_shape_is_bitwise_neutral(monkeypatch, handles, N, cart, k):
    """RSLAM_CHOL_OUTER_SMALL=0 (128 x 64 tiles for the Cholesky's K = 256 updates) gives the same bits as the default 64 x 64 tiles."""
    _, xa, Pa = single(monkeypatch, handles, N, k, cart=cart)
    hb, xb, Pb = single(monkeypatch, handles, N, k, cart=cart, env={"RSLAM_CHOL_OUTER_SMALL": 0})
    assert set(hb.route()[1]["chol_outer"]) == {(128, 64)}
    assert np.array_equal(xa, xb) and np.array_equal(Pa, Pb)
