"""nk_index_kmeanspp (k-means++ seeding over every row, on the device) against the sequential reference loop of
kmeans.go:364-427 (kmeanspp_ref.c) with the same injected random numbers.  Every comparison reports, on a mismatch, how far
that step's target lay from the nearest cumulative boundary, so a rounding tie is told apart from a wrong selection.
Integer-valued rows make every sum exact: there the device must agree bit for bit."""
import ctypes as C

import numpy as np
import pytest

import kmeanspp_ref

pytestmark = pytest.mark.gpu


def _mixture(rng, n, d, m, sigma):
    mu = rng.uniform(-1, 1, (m, d)).astype(np.float32)
    return (mu[rng.integers(0, m, n)] + rng.standard_normal((n, d)).astype(np.float32) * np.float32(sigma)).astype(np.float32)


def _index(rows, devices=(0,)):
    from nornicdb_b200.knn import KnnIndex
    ix = KnnIndex(rows.shape[1], metric="euclidean", devices=devices)
    ix.upload(rows)
    return ix


def _seed(ix, rows, K, first, draws):
    cen, picked, scored = ix.kmeanspp(K, first, draws)
    wc, wp = kmeanspp_ref.seq(rows, K, first, draws)
    assert (picked == wp).all(), kmeanspp_ref.explain(picked, wp, rows, draws)
    np.testing.assert_array_equal(cen, wc)
    np.testing.assert_array_equal(cen, rows[picked])
    return picked, scored


PARITY = [  # (n, d, K)
    (1, 3, 1), (2, 32, 2), (7, 100, 7), (50, 3, 50), (257, 100, 257), (1000, 3, 17), (1500, 128, 100), (5000, 100, 100),
    (20_000, 1024, 17), (40_000, 32, 100), (300_000, 3, 100), (300_001, 32, 17),
]


@pytest.mark.parametrize("kind", ["uniform", "mixture"])
@pytest.mark.parametrize("n,d,K", PARITY)
def test_parity_with_the_sequential_loop(knn_lib, gpu_device, kind, n, d, K):
    rng = np.random.default_rng(n * 7 + d + K)
    rows = rng.uniform(-1, 1, (n, d)).astype(np.float32) if kind == "uniform" else _mixture(rng, n, d, 20, 0.05)
    ix = _index(rows)
    launches = ix.stats()["kernel_launches"]
    first = int(rng.integers(n))
    _, scored = _seed(ix, rows, K, first, rng.random(K - 1))
    assert 0 < scored <= max(K - 1, 1) * n if K > 1 else scored == 0
    assert ix.stats()["kernel_launches"] - launches == (0 if K == 1 else 1 + (K - 1) + 2 * (K - 2))
    ix.release()


def _int_rows(rng, n, d, lo=-4, hi=5):
    return rng.integers(lo, hi, (n, d)).astype(np.float32)


def test_boundary_draws_select_that_row(knn_lib, gpu_device):
    rng = np.random.default_rng(1)
    rows = _int_rows(rng, 3000, 5)
    ix = _index(rows)
    d2 = ((rows - rows[17]).astype(np.float64) ** 2).sum(1)
    cum, total = np.cumsum(d2), d2.sum()
    tried = 0
    for i in rng.choice(np.flatnonzero(d2 > 0), 60, replace=False):
        u = cum[i] / total
        if u >= 1.0 or u * total != cum[i]:
            continue  # only targets that are exactly the cumulative sum of row i
        picked, _ = _seed(ix, rows, 2, 17, [u])
        assert picked[1] == i
        tried += 1
    assert tried >= 20
    ix.release()


@pytest.mark.parametrize("case", ["u0", "identical", "duplicates", "nan", "inf", "integers"])
def test_exact_semantics_on_integer_rows(knn_lib, gpu_device, case):
    rng = np.random.default_rng(len(case))
    n, d, K = 5000, 12, 40
    rows = _int_rows(rng, n, d)
    draws = rng.random(K - 1)
    first = int(rng.integers(n))
    if case == "u0":
        draws[:] = 0.0
    elif case == "identical":
        rows[:] = 3.0
    elif case == "duplicates":
        rows = np.tile(_int_rows(rng, 50, d, 0, 3), (n // 50, 1))
    elif case == "nan":
        rows[1234, 3] = np.nan
        first = 10
    elif case == "inf":
        rows[4321, 0] = np.inf
        first = 10
    ix = _index(rows)
    picked, _ = _seed(ix, rows, K, first, draws)
    if case == "u0":
        assert (picked[1:] == 0).all()       # cumWeight >= 0 at row 0
    if case == "identical":
        assert (picked[1:] == 0).all()       # total 0 -> target 0 -> row 0, again and again
    if case == "nan":
        assert (picked[1:] == n - 1).all()   # NaN total: no cumulative sum reaches the target
    if case == "inf":
        assert picked[1] == 4321             # infinite weight, selected as soon as the sum reaches inf
    again = ix.kmeanspp(K, first, draws)     # determinism: bit-identical on a second call
    np.testing.assert_array_equal(again[1], picked)
    ix.release()


@pytest.mark.parametrize("inf_row", [700_000, 700_416, 1_099_999])
def test_inf_row_where_each_select_thread_sums_several_blocks(knn_lib, gpu_device, inf_row):
    # > 1024 blocks of 1024 rows: a select thread owns a run of blocks, and the Inf may start, sit inside or end the run
    rng = np.random.default_rng(inf_row)
    rows = _int_rows(rng, 1_100_000, 4)
    rows[inf_row, 2] = np.inf
    ix = _index(rows)
    picked, _ = _seed(ix, rows, 4, 3, rng.random(3))
    assert picked[1] == inf_row
    ix.release()


def test_skip_bound_engages_on_separated_mixture(knn_lib, gpu_device):
    rng = np.random.default_rng(3)
    n, d, K = 200_000, 32, 100
    rows = _mixture(rng, n, d, 50, 0.01)
    ix = _index(rows)
    draws = rng.random(K - 1)
    picked, scored = _seed(ix, rows, K, 5, draws)
    assert scored < 0.5 * (K - 1) * n, scored / ((K - 1) * n)
    a = ix.kmeanspp(K, 5, draws)
    b = ix.kmeanspp(K, 5, draws)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
    assert a[2] == scored
    ix.release()


def test_skip_bound_with_equidistant_rows(knn_lib, gpu_device):
    # a symmetric lattice: many rows are exactly as far from the new centroid as from the old one (strict < keeps them)
    g = np.arange(-3, 4, dtype=np.float32)
    lattice = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    rows = np.concatenate([lattice, lattice * 2, -lattice]).astype(np.float32)
    rng = np.random.default_rng(4)
    ix = _index(rows)
    for trial in range(4):
        K = 60
        _seed(ix, rows, K, int(rng.integers(rows.shape[0])), rng.random(K - 1))
    ix.release()


@pytest.mark.parametrize("kind", ["integers", "mixture"])
def test_three_shards_on_one_gpu_equal_one_shard(knn_lib, gpu_device, kind):
    rng = np.random.default_rng(6)
    n, d, K = 30_001, 64, 50
    rows = _int_rows(rng, n, d) if kind == "integers" else _mixture(rng, n, d, 30, 0.05)
    draws = rng.random(K - 1)
    one = _index(rows)
    three = _index(rows, devices=(0, 0, 0))
    for first in (0, 15_000, n - 1):
        a = one.kmeanspp(K, first, draws)
        b = three.kmeanspp(K, first, draws)
        assert (a[1] == b[1]).all(), kmeanspp_ref.explain(b[1], a[1], rows, draws)
        np.testing.assert_array_equal(a[0], b[0])
        assert a[2] == b[2]
    _seed(three, rows, K, 7, draws)
    one.release()
    three.release()


def test_real_multi_gpu(knn_lib, gpu_device):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    rng = np.random.default_rng(8)
    rows = _mixture(rng, 50_000, 128, 40, 0.05)
    ix = _index(rows, devices=tuple(range(torch.cuda.device_count())))
    _seed(ix, rows, 64, 3, rng.random(63))
    ix.release()


def test_errors_leave_the_index_usable(knn_lib, gpu_device):
    from nornicdb_b200 import _lib
    from nornicdb_b200.knn import KnnError, KnnIndex
    rng = np.random.default_rng(9)
    rows = rng.standard_normal((100, 16)).astype(np.float32)
    ix = _index(rows)
    with pytest.raises(KnnError, match="K must be"):
        ix.kmeanspp(0, 0, [])
    with pytest.raises(KnnError, match="exceeds"):
        ix.kmeanspp(101, 0, rng.random(100))
    with pytest.raises(KnnError, match="first_row"):
        ix.kmeanspp(3, 100, rng.random(2))
    cen = np.empty((3, 16), np.float32)
    assert ix.lib.nk_index_kmeanspp(ix.ptr, 3, 0, None, cen.ctypes.data_as(C.c_void_p), None, None) == -1
    assert "draws" in _lib.last_error()
    h = KnnIndex(16, metric="euclidean", dtype="f16")
    h.upload(rows.astype(np.float16))
    with pytest.raises(KnnError, match="fp32"):
        h.kmeanspp(3, 0, rng.random(2))
    h.release()
    _seed(ix, rows, 10, 4, rng.random(9))  # still usable
    ix.release()


def test_cluster_index_seeds_on_the_device_like_the_host(knn_lib, gpu_device):
    from nornicdb_b200.cluster_index import ClusterIndex, KMeansConfig
    rng = np.random.default_rng(10)
    n, d, K = 4000, 8, 20
    rows = _int_rows(rng, n, d, -3, 4)
    cfg = KMeansConfig(NumClusters=K, AutoK=False)
    dev = ClusterIndex(d, cfg, rng=np.random.default_rng(77))
    dev.AddBatch([f"n{i}" for i in range(n)], rows)
    dev.Cluster()
    host = ClusterIndex(d, cfg, rng=np.random.default_rng(77))
    host.AddBatch([f"n{i}" for i in range(n)], rows)
    init = host._init_kmeanspp(K, host._ix.read_rows(0, n))
    host.Cluster(initial_centroids=init)
    np.testing.assert_array_equal(dev.centroids, host.centroids)
    np.testing.assert_array_equal(dev.assignments, host.assignments)
    # a multi-device ClusterIndex clusters end to end, with the same result on integer rows
    multi = ClusterIndex(d, cfg, devices=(0, 0), rng=np.random.default_rng(77))
    multi.AddBatch([f"n{i}" for i in range(n)], rows)
    multi.Cluster()
    assert multi.IsClustered() and multi.NumClusters() == K
    np.testing.assert_array_equal(multi.centroids, dev.centroids)
    np.testing.assert_array_equal(multi.assignments, dev.assignments)
    for ci in (dev, host, multi):
        ci.Clear()


def test_large_shape_against_torch_fp64(knn_lib, gpu_device):
    """2M x 1024 mixture, K = 1000, against an independent torch fp64 restatement of the loop on the same GPU."""
    import torch
    from nornicdb_b200.knn import KnnIndex
    n, d, K = 2_000_000, 1024, 1000
    ix = KnnIndex(d, metric="euclidean")
    ix.fill_clustered(n, seed=5, n_centres=1000, sigma=0.1)
    rng = np.random.default_rng(12)
    first, draws = int(rng.integers(n)), rng.random(K - 1)
    cen, picked, scored = ix.kmeanspp(K, first, draws)
    X = torch.from_numpy(ix.read_rows(0, n)).cuda()
    ix.release()

    def dist(c):
        out = torch.empty(n, dtype=torch.float64, device="cuda")
        for s in range(0, n, 1 << 18):
            out[s:s + (1 << 18)] = (X[s:s + (1 << 18)] - c).double().square().sum(1)
        return out

    mind = dist(X[first])
    want, margins = [first], []
    for c in range(1, K):
        total = mind.sum()
        cum = torch.cumsum(mind, 0)
        target = float(draws[c - 1]) * total
        sel = min(int(torch.searchsorted(cum, target.reshape(1)).item()), n - 1)
        margins.append(float((cum - target).abs().min() / total))
        want.append(sel)
        if sel != int(picked[c]):
            break  # from here on the two runs seed from different centroids
        if c + 1 < K:
            mind = torch.minimum(mind, dist(X[sel]))
    want = np.array(want)
    bad = np.flatnonzero(want != picked[:len(want)])
    print(f"large shape: rows_scored / ((K-1) n) = {scored / ((K - 1) * n):.4f}, smallest target margin {min(margins):.3e}")
    if bad.size:
        c = int(bad[0])
        assert margins[c - 1] < 1e-12, f"step {c}: device {picked[c]}, torch {want[c]}, margin {margins[c - 1]:.3e}"
    else:
        assert len(want) == K
        np.testing.assert_array_equal(cen, X[torch.from_numpy(picked.astype(np.int64)).cuda()].cpu().numpy())
