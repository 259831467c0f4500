"""Edges of k_gemm_dmma's copy path: per-tile row tests and source pointers, and the last k-chunk peeled off with its column test.

Each case runs one joint update through tests/test_gpu_update_kernels.py's Handle (float64 reference at its bar, P exactly
symmetric, launches as route() says) on shapes that put the edges under the GEMM's operands:
  * K mod 16 in {2, 14, 0}: the syrk_P K (= k) and the Cholesky's K = 256 outer updates over a trailing size k - o of the same
    residues; the TRSM's K = 1024 outer GEMMs with k - 1024 of those residues;
  * n + 1 one above and one below a multiple of 128 (the 128 x 64 syrk_P / trsm_outer tiles) and of 64 (the 64 x 64 syrk_P tiles);
  * leading dimensions larger than the map (a handle sized for more features);
  * a batch of two maps of different sizes.
Map sizes: n + 1 = 14 + 6 N - 3 c for N features of which c are cartesian."""
import pytest

from tests.test_gpu_update_kernels import Handle, single


@pytest.fixture
def handles():
    made = []
    yield made
    for h in made:
        h.close()


# (N, cartesian positions) -> n + 1
MAPS = {
    "n1-128a+1": (553, (552,)),   # n + 1 = 3329 = 26 * 128 + 1
    "n1-128a-1": (574, (573,)),   # n + 1 = 3455 = 27 * 128 - 1
    "n1-64a+1": (521, (520,)),    # n + 1 = 3137 = 49 * 64 + 1
    "n1-64a-1": (542, (541,)),    # n + 1 = 3263 = 51 * 64 - 1
}


def n_plus_1(N, cart):
    return 14 + 6 * N - 3 * len(cart)


def test_map_table_sits_on_the_edges():
    """The table's maps have the n + 1 their names say (no GPU needed)."""
    assert [n_plus_1(*m) for m in MAPS.values()] == [26 * 128 + 1, 27 * 128 - 1, 49 * 64 + 1, 51 * 64 - 1]
    assert n_plus_1(137, (136,)) == 13 * 64 + 1 and n_plus_1(158, (157,)) == 15 * 64 - 1


@pytest.mark.gpu
@pytest.mark.parametrize("k", [258, 270, 272, 1038, 1040, 1042])
@pytest.mark.parametrize("shape", list(MAPS))
def test_k_residues_on_row_edges(monkeypatch, handles, shape, k):
    """k mod 16 = 2, 14, 0 (k - 1024 as well for the TRSM's outer GEMM) on maps whose n + 1 sits next to a tile multiple."""
    N, cart = MAPS[shape]
    h, _, _ = single(monkeypatch, handles, N, k, cart=cart)
    _, v = h.route()
    assert v["syrk_P"] == (128, 64) and v["trsm_outer_at"] == [1024]  # launched for kmax = 2 N; it has work when k > 1024


@pytest.mark.gpu
@pytest.mark.parametrize("N,cart,k", [(137, (136,), 258), (137, (136,), 270), (158, (157,), 272), (158, (157,), 302)],
                         ids=["n833-k258", "n833-k270", "n959-k272", "n959-k302"])
def test_small_tiles_on_row_edges(monkeypatch, handles, N, cart, k):
    """k_gemm_dmma<64, 64> syrk_P with n + 1 one above / below a multiple of 64 and k mod 16 = 2, 14, 0."""
    h, _, _ = single(monkeypatch, handles, N, k, cart=cart)
    assert h.route()[1]["syrk_P"] == (64, 64)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [270, 1038])
def test_leading_dimensions_larger_on_row_edges(monkeypatch, handles, k):
    """n + 1 = 26 * 128 + 1 on a handle sized for 700 features: ldp / ldw / lds larger than the map needs."""
    N, cart = MAPS["n1-128a+1"]
    single(monkeypatch, handles, N, k, cart=cart, max_features=700)


@pytest.mark.gpu
def test_batch_of_row_edge_maps(monkeypatch, handles):
    """B = 2: n + 1 = 27 * 128 - 1 and 26 * 128 + 1 on one handle with k = (1038, 270), then (272, 1042) on the updated covariances."""
    h = Handle(monkeypatch, 574, batch=2)
    handles.append(h)
    h.upload(0, *MAPS["n1-128a-1"])
    h.upload(1, *MAPS["n1-128a+1"])
    h.update(0, {0: h.linearise(0, 1038, 0), 1: h.linearise(1, 270, 0)})
    h.update(0, {0: h.linearise(0, 272, 0, lin_seed=1), 1: h.linearise(1, 1042, 0, lin_seed=1)})
