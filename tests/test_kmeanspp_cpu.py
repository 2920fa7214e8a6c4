"""k-means++ seeding without a GPU: the sequential reference loop (kmeanspp_ref.c) against a line-for-line Python
transliteration of kmeans.go:364-427, and ClusterIndex.Cluster's choice of seeding over index stand-ins with and without
`kmeanspp` (which draws it consumes, in which order, and that "random" and initial_centroids are left alone)."""
import numpy as np
import pytest

import kmeanspp_ref
from fake_knn import FakeKnnIndex


def _cases():
    rng = np.random.default_rng(11)
    yield "uniform", rng.uniform(-1, 1, (40, 5)).astype(np.float32), 7
    yield "uniform-d8", rng.standard_normal((33, 8)).astype(np.float32), 33  # K = n
    yield "integers", rng.integers(-3, 4, (50, 3)).astype(np.float32), 12
    yield "identical", np.ones((9, 4), dtype=np.float32), 5                  # total 0: row 0 repeats
    dup = rng.integers(0, 3, (6, 2)).astype(np.float32)
    yield "duplicates", np.concatenate([dup, dup, dup]), 8
    nan = rng.integers(0, 5, (20, 3)).astype(np.float32)
    nan[4, 1] = np.nan
    yield "nan-row", nan, 5                                                  # n - 1 from then on
    inf = rng.integers(0, 5, (20, 3)).astype(np.float32)
    inf[11, 0] = np.inf
    yield "inf-row", inf, 4
    yield "one-row", rng.standard_normal((1, 6)).astype(np.float32), 1


@pytest.mark.parametrize("name,rows,K", list(_cases()), ids=[c[0] for c in _cases()])
def test_sequential_reference_matches_the_transliteration(name, rows, K):
    rng = np.random.default_rng(len(name))
    for trial in range(3):
        first = int(rng.integers(rows.shape[0]))
        draws = rng.random(K - 1)
        if trial == 2 and K > 1:
            draws[0] = 0.0  # u = 0: the first row with a positive cumulative weight (or row 0)
        cen, picked = kmeanspp_ref.seq(rows, K, first, draws)
        want = kmeanspp_ref.transliteration(rows, K, first, draws)
        assert picked.tolist() == want, (name, trial)
        np.testing.assert_array_equal(cen, rows[want])
        if name == "identical":
            assert want[1:] == [0] * (K - 1)
        if name == "nan-row":
            assert want[1:] == [rows.shape[0] - 1] * (K - 1)
        if name == "inf-row" and first != 11:
            assert want[1] == (11 if draws[0] > 0 else rows.shape[0] - 1)  # u * inf = inf reaches row 11; 0 * inf = NaN


def test_boundary_draw_selects_that_row():
    rows = np.array([[0, 0], [1, 0], [0, 2], [3, 0], [0, 0]], dtype=np.float32)  # D2 from row 0: 0 1 4 9 0, total 14
    for i, cum in ((1, 1.0), (2, 5.0), (3, 14.0)):
        u = cum / 14.0
        assert u * 14.0 == cum  # the target is exactly the cumulative sum of row i
        _, picked = kmeanspp_ref.seq(rows, 2, 0, [u])
        assert picked[1] == i and kmeanspp_ref.transliteration(rows, 2, 0, [u])[1] == i


class FakeSeedingKnnIndex(FakeKnnIndex):
    """FakeKnnIndex + a `kmeanspp` that runs the sequential reference and records what it was given."""

    def kmeanspp(self, K, first_row, draws):
        self.seed_calls = getattr(self, "seed_calls", []) + [(int(K), int(first_row), np.array(draws, dtype=np.float64))]
        cen, picked = kmeanspp_ref.seq(self._rows.astype(np.float32), int(K), int(first_row), draws)
        return cen, picked, int(K) * len(self)


def _index(monkeypatch, cls, rows, seed, **cfg):
    import nornicdb_b200.embedding_index as ei
    from nornicdb_b200.cluster_index import ClusterIndex, KMeansConfig
    monkeypatch.setattr(ei, "KnnIndex", cls)
    ci = ClusterIndex(rows.shape[1], KMeansConfig(**cfg), rng=np.random.default_rng(seed))
    ci.AddBatch([f"n{i}" for i in range(rows.shape[0])], rows)
    return ci


@pytest.fixture()
def small_int_rows():
    rng = np.random.default_rng(5)
    return rng.integers(-4, 5, (300, 6)).astype(np.float32)


def test_device_seeding_consumes_the_host_draws_in_order(monkeypatch, oracle_mod, small_int_rows):
    rows, K = small_int_rows, 9
    ci = _index(monkeypatch, FakeSeedingKnnIndex, rows, 21, NumClusters=K, AutoK=False)
    ci.Cluster()
    (k, first, draws), = ci._ix.seed_calls
    ref = np.random.default_rng(21)
    assert k == K and first == int(ref.integers(rows.shape[0]))
    np.testing.assert_array_equal(draws, ref.random(K - 1))
    # same rng, host seeding on the rows read back: the same draws pick the same rows on integer data
    host = _index(monkeypatch, FakeKnnIndex, rows, 21, NumClusters=K, AutoK=False)
    init = host._init_kmeanspp(K, host._ix.read_rows(0, rows.shape[0]))
    np.testing.assert_array_equal(init, kmeanspp_ref.seq(rows, K, first, draws)[0])
    again = _index(monkeypatch, FakeKnnIndex, rows, 99, NumClusters=K, AutoK=False)
    again.Cluster(initial_centroids=init)
    np.testing.assert_array_equal(ci.centroids, again.centroids)
    np.testing.assert_array_equal(ci.assignments, again.assignments)


def test_host_seeding_without_kmeanspp(monkeypatch, oracle_mod, small_int_rows):
    rows, K = small_int_rows, 7
    ci = _index(monkeypatch, FakeKnnIndex, rows, 3, NumClusters=K, AutoK=False)
    assert not hasattr(ci._ix, "kmeanspp")
    ci.Cluster()
    twin = _index(monkeypatch, FakeKnnIndex, rows, 3, NumClusters=K, AutoK=False)
    init = twin._init_kmeanspp(K, rows)
    ref = _index(monkeypatch, FakeKnnIndex, rows, 0, NumClusters=K, AutoK=False)
    ref.Cluster(initial_centroids=init)
    np.testing.assert_array_equal(ci.centroids, ref.centroids)
    np.testing.assert_array_equal(ci.assignments, ref.assignments)


def test_random_init_and_initial_centroids_do_not_seed_on_the_device(monkeypatch, oracle_mod, small_int_rows):
    rows, K = small_int_rows, 5
    ci = _index(monkeypatch, FakeSeedingKnnIndex, rows, 8, NumClusters=K, AutoK=False, InitMethod="random")
    ci.Cluster()
    assert not hasattr(ci._ix, "seed_calls")
    twin = _index(monkeypatch, FakeKnnIndex, rows, 8, NumClusters=K, AutoK=False, InitMethod="random")
    twin.Cluster()
    np.testing.assert_array_equal(ci.centroids, twin.centroids)
    given = _index(monkeypatch, FakeSeedingKnnIndex, rows, 8, NumClusters=K, AutoK=False)
    given.Cluster(initial_centroids=rows[:K])
    assert not hasattr(given._ix, "seed_calls")
    ref = _index(monkeypatch, FakeKnnIndex, rows, 1, NumClusters=K, AutoK=False)
    ref.Cluster(initial_centroids=rows[:K])
    np.testing.assert_array_equal(given.centroids, ref.centroids)
