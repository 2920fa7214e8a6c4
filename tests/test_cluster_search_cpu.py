"""ClusterIndex's routed search over a CPU stand-in of the device index (tests/fake_knn.py plus a numpy restatement of
nk_index_set_clusters / nk_search_clusters): lazy installation of the clustering, the two cases served on the host, batch vs
single-query results, error identities."""
import numpy as np
import pytest

import oracle
from fake_knn import FakeKnnIndex
from nornicdb_b200.knn import KnnError


class FakeClusterKnnIndex(FakeKnnIndex):
    """FakeKnnIndex + the routed search: route (float32 differences, float64 squares, stable by id), members in (probe
    rank, row) order, exact fp64 scores, ties by candidate position, sentinel padding to min(k, rows).  Row-count changing
    mutations drop the clustering, as on the device."""

    _clusters = None

    def upload(self, rows):
        super().upload(rows)
        self._clusters = None

    def append(self, rows):
        super().append(rows)
        self._clusters = None

    def remove_swap(self, row):
        super().remove_swap(row)
        self._clusters = None

    def set_clusters(self, centroids, assign):
        if centroids is None:
            self._clusters = None
            return
        a = np.asarray(assign, dtype=np.int64).reshape(-1)
        if a.size != len(self):
            raise KnnError("assignments do not cover the rows")
        self._clusters = (np.array(centroids, dtype=np.float32), a.copy())
        self.cluster_installs = getattr(self, "cluster_installs", 0) + 1

    def search_clusters(self, queries, k, n_probe, return_probes=False):
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32)).reshape(-1, self.dim)
        if self._clusters is None:
            raise KnnError("nk_search_clusters: no clusters set")
        if k > 1024 or n_probe <= 0:
            raise KnnError("bad k / n_probe")
        cen, assign = self._clusters
        self.searches += 1
        ke, P = min(int(k), len(self)), min(int(n_probe), cen.shape[0])
        idx = np.full((q.shape[0], ke), 0xFFFFFFFF, np.uint32)
        sc = np.zeros((q.shape[0], ke), np.float32)
        probes = np.empty((q.shape[0], P), np.int32)
        for i, v in enumerate(q):
            d = ((cen - v[None, :]).astype(np.float64) ** 2).sum(1)
            probes[i] = np.argsort(d, kind="stable")[:P]
            cand = np.concatenate([np.nonzero(assign == c)[0] for c in probes[i]])
            if self._mask is not None:
                cand = cand[self._mask[cand]]
            n = min(ke, len(cand))
            if n:
                o_i, o_s = oracle.knn_exact64(self._rows[cand], v.reshape(1, -1), n, self.metric)
                idx[i, :n], sc[i, :n] = cand[o_i[0]], o_s[0]
        return (idx, sc, probes) if return_probes else (idx, sc)


@pytest.fixture()
def clustered(monkeypatch, oracle_mod):
    import nornicdb_b200.embedding_index as ei
    from nornicdb_b200.cluster_index import ClusterIndex, KMeansConfig
    monkeypatch.setattr(ei, "KnnIndex", FakeClusterKnnIndex)
    rng = np.random.default_rng(4)
    mu = rng.uniform(-1, 1, (8, 24)).astype(np.float32)
    rows = (mu[rng.integers(0, 8, 500)] + rng.standard_normal((500, 24)).astype(np.float32) * 0.1).astype(np.float32)
    ci = ClusterIndex(24, KMeansConfig(NumClusters=8, AutoK=False), rng=np.random.default_rng(1))
    ci.AddBatch([f"n{i}" for i in range(500)], rows)
    ci.Cluster()
    return ci, rows


def _ids(res):
    return None if res is None else [(r.ID, round(r.Score, 6), round(r.Distance, 6)) for r in res]


def test_routed_search_matches_the_host_path_and_batches(clustered):
    ci, rows = clustered
    for nc in (1, 3, 8, 20):
        for topK in (1, 5, 100, 600):
            batch = ci.SearchWithClustersBatch(rows[:6], topK, nc)
            for i in range(6):
                one = ci.SearchWithClusters(rows[i], topK, nc)
                assert _ids(one) == _ids(batch[i])
                assert _ids(one) == _ids(ci._search_with_clusters_host(rows[i], topK, nc))
    assert ci.SearchWithClusters(rows[0], 0, 3) == []        # topK <= 0 with candidates: empty list
    assert ci.SearchWithClusters(rows[0], 5, 0) is None      # no clusters routed: nil
    with pytest.raises(ValueError):
        ci.SearchWithClusters(rows[0][:10], 5, 2)            # ErrInvalidDimensions
    from nornicdb_b200.cluster_index import ErrInvalidDimensions
    with pytest.raises(ErrInvalidDimensions):
        ci.SearchWithClustersBatch(rows[:2, :10], 5, 2)


def test_clustering_is_reinstalled_lazily(clustered):
    ci, rows = clustered
    ix = ci._ix
    ci.SearchWithClusters(rows[0], 5, 2)
    ci.SearchWithClustersBatch(rows[:4], 5, 2)
    assert ix.cluster_installs == 1                           # installed once, reused
    ci.OnNodeUpdate("n3", rows[200])
    ci.SearchWithClusters(rows[0], 5, 2)
    assert ix.cluster_installs == 2
    np.testing.assert_array_equal(ix._clusters[1], ci.assignments)
    ci.UpdateCentroidsBatch()
    ci.SearchWithClusters(rows[0], 5, 2)
    assert ix.cluster_installs == 3
    np.testing.assert_array_equal(ix._clusters[0], ci.centroids)
    ci.Cluster()
    ci.SearchWithClusters(rows[0], 5, 2)
    assert ix.cluster_installs == 4
    ci.OnNodeUpdate("fresh", rows[7])                         # a new row: the device dropped the clustering, re-installed
    res = ci.SearchWithClusters(rows[7], 3, 1)
    assert ix.cluster_installs == 5 and {r.ID for r in res[:2]} == {"n7", "fresh"}
    ci.Clear()
    assert ci.SearchWithClusters(rows[0], 5, 2) is None       # not clustered, empty: Search -> nil


def test_host_path_cases(clustered, monkeypatch):
    ci, rows = clustered
    want = _ids(ci._search_with_clusters_host(rows[1], 1500, 8))

    def no_device(*a, **kw):
        raise AssertionError("served on the device")
    monkeypatch.setattr(ci._ix, "search_clusters", no_device)
    assert _ids(ci.SearchWithClusters(rows[1], 1500, 8)) == want and len(want) == 500   # topK > NK_MAX_K
    ci.Add("extra", rows[3])                                  # Add without OnNodeUpdate: the assignments no longer cover
    assert len(ci.assignments) != ci.Count()                  # the rows exactly
    got = ci.SearchWithClustersBatch(rows[:3], 5, 2)
    assert [_ids(g) for g in got] == [_ids(ci._search_with_clusters_host(v, 5, 2)) for v in rows[:3]]


def test_index_without_routed_search_takes_the_subset_path(monkeypatch, oracle_mod):
    """An index back-end that only scores subsets (the plain CPU stand-in) answers through the reference's own path."""
    import nornicdb_b200.embedding_index as ei
    from nornicdb_b200.cluster_index import ClusterIndex, KMeansConfig
    monkeypatch.setattr(ei, "KnnIndex", FakeKnnIndex)
    rng = np.random.default_rng(9)
    rows = rng.standard_normal((200, 16)).astype(np.float32)
    ci = ClusterIndex(16, KMeansConfig(NumClusters=4, AutoK=False), rng=np.random.default_rng(2))
    ci.AddBatch([f"n{i}" for i in range(200)], rows)
    ci.Cluster()
    assert [_ids(r) for r in ci.SearchWithClustersBatch(rows[:3], 7, 2)] == [_ids(ci._search_with_clusters_host(v, 7, 2)) for v in rows[:3]]
