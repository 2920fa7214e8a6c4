"""Cluster-routed search (nk_index_set_clusters + nk_search_clusters[_device]) against an fp64 brute force restricted to each
query's candidate set: routing, the metric x dtype x shape grid, cross-checks with nk_search / nk_score_subset, adversarial
cluster shapes, front-end semantics, lifecycle, the device-resident form, and one large clustered corpus."""
import numpy as np
import pytest

from parity import check_parity, exact_scores_for

pytestmark = pytest.mark.gpu

SENT = 0xFFFFFFFF


def _mixture(n, d, centres, seed, sigma=0.15):
    rng = np.random.default_rng(seed)
    mu = rng.uniform(-1, 1, (centres, d)).astype(np.float32)
    lab = rng.integers(0, centres, n)
    return (mu[lab] + rng.standard_normal((n, d)).astype(np.float32) * sigma).astype(np.float32), mu


def _route(cen, q, P):
    d = np.concatenate([((cen[None, :, :] - q[i:i + 16, None, :]).astype(np.float64) ** 2).sum(-1)  # float32 differences,
                        for i in range(0, q.shape[0], 16)])                                          # float64 squares
    return np.argsort(d, axis=1, kind="stable")[:, :P], d


def _check_probes(cen, q, got):
    """Probe lists equal the host restatement; a different cluster only where the fp64 distances tie within 2e-6."""
    want, d = _route(cen, q, got.shape[1])
    swaps = 0
    for i in range(q.shape[0]):
        for r in np.nonzero(got[i] != want[i])[0]:
            a, b = d[i, got[i, r]], d[i, want[i, r]]
            assert abs(a - b) <= 2e-6 * max(a, b, 1e-30), (i, r, got[i], want[i], a, b)
            swaps += 1
    return swaps


def _candidates(assign, probes):
    return np.concatenate([np.nonzero(assign == c)[0] for c in probes]) if len(probes) else np.empty(0, np.int64)


def _oracle(rows, cen, assign, q, k, P, metric, mask=None, floor=None):
    """fp64 brute force over each query's candidates, ties by candidate position; rows beyond the candidates -> sentinel."""
    probes, _ = _route(cen, q, P)
    out_i, out_s = [], []
    for i in range(q.shape[0]):
        cand = _candidates(assign, probes[i])
        if mask is not None:
            cand = cand[mask[cand]]
        s = exact_scores_for(rows, q[i], cand, metric)
        order = np.lexsort((np.arange(len(cand)), s if metric == "euclidean" else -s))
        if floor is not None:
            order = order[(s[order] <= floor) if metric == "euclidean" else (s[order] >= floor)]
        out_i.append(cand[order[:k]])
        out_s.append(s[order[:k]])
    return out_i, out_s


def _compare(rows, q, metric, gi, gs, oi, os_):
    swaps = 0
    for i in range(q.shape[0]):
        n = len(oi[i])
        assert (gi[i, n:] == SENT).all() and (gs[i, n:] == 0).all(), (i, n, gi[i])
        assert (gi[i, :n] != SENT).all(), (i, n, gi[i])
        if n:
            swaps += check_parity(rows, q[i:i + 1], n, metric, gi[i:i + 1, :n], gs[i:i + 1, :n], oi[i][None, :], os_[i][None, :])
    return swaps


def _index(rows, metric, dtype="f32"):
    from nornicdb_b200.knn import KnnIndex
    ix = KnnIndex(rows.shape[1], metric=metric, dtype=dtype)
    ix.upload(rows)
    return ix


def _stored(ix, rows):
    """The rows as the index holds them (fp16 / bf16 rounding), as fp32."""
    from nornicdb_b200.knn import from_bf16_bits
    back = ix.read_rows(0, rows.shape[0])
    return from_bf16_bits(back) if ix.dtype == 2 else back.astype(np.float32)


def test_routing_matches_the_host_restatement(knn_lib):
    rows, mu = _mixture(3000, 64, 40, 1)
    cen = (mu + 0.01).astype(np.float32)
    cen[7] = cen[3]                                  # duplicate centroids: the lower id wins
    cen[8] = cen[3]
    assign = np.arange(3000, dtype=np.int32) % 40
    ix = _index(rows, "cosine")
    ix.set_clusters(cen, assign)
    rng = np.random.default_rng(2)
    q = rng.uniform(-1, 1, (300, 64)).astype(np.float32)
    q[0] = 0.0                                       # zero query
    q[1] = cen[3]                                    # exactly on the duplicated centroid
    swaps = 0
    for P in (1, 3, 10, 40, 99):                     # n_probe > K is clamped to K
        _, _, probes = ix.search_clusters(q, 5, P, return_probes=True)
        assert probes.shape == (300, min(P, 40))
        swaps += _check_probes(cen, q, probes)
        assert list(probes[1, :3]) == [3, 7, 8][:probes.shape[1]]
    assert swaps <= 3
    one = _index(rows[:500], "dot")
    one.set_clusters(cen[:1], np.zeros(500, np.int32))  # K = 1: every query probes cluster 0
    i1, s1, p1 = one.search_clusters(q[:7], 10, 3, return_probes=True)
    assert p1.shape == (7, 1) and (p1 == 0).all()
    oi, os_ = _oracle(rows[:500], cen[:1], np.zeros(500), q[:7], 10, 1, "dot")
    _compare(rows[:500], q[:7], "dot", i1, s1, oi, os_)
    ix.release(); one.release()


GRID = [  # (metric, dtype, d, Q, k, n_probe)
    ("cosine", "f32", 128, 1, 10, 3), ("cosine", "f32", 1024, 64, 100, 3), ("cosine", "f16", 30, 7, 1, 10),
    ("cosine", "bf16", 128, 300, 10, 1), ("dot", "f32", 30, 300, 1024, 3), ("dot", "f16", 1024, 7, 10, 10),
    ("dot", "bf16", 1024, 1, 100, 3), ("euclidean", "f32", 128, 1024, 10, 3), ("euclidean", "f16", 128, 64, 1024, 1),
    ("euclidean", "bf16", 30, 64, 10, 50), ("cosine", "f32", 30, 1024, 100, 50), ("dot", "f32", 128, 7, 10, 50),
]


@pytest.mark.parametrize("metric,dtype,d,Q,k,n_probe", GRID)
def test_results_across_the_grid(knn_lib, metric, dtype, d, Q, k, n_probe):
    K = 50
    rows, mu = _mixture(12_000, d, K, 3 + d)
    assign = np.random.default_rng(d).integers(0, K, rows.shape[0]).astype(np.int32)
    assign[::97] = np.argmin(((rows[::97, None, :] - mu[None]) ** 2).sum(-1), 1)
    ix = _index(rows, metric, dtype)
    stored = _stored(ix, rows)
    ix.set_clusters(mu, assign)
    q = (rows[np.random.default_rng(5).integers(0, rows.shape[0], Q)] + 0.05).astype(np.float32)
    gi, gs, probes = ix.search_clusters(q, k, n_probe, return_probes=True)
    assert gi.shape == (Q, k)
    _check_probes(mu, q, probes)
    oi, os_ = _oracle(stored, mu, assign, q, k, min(n_probe, K), metric)
    assert _compare(stored, q, metric, gi, gs, oi, os_) <= max(4, Q * k // 500)  # fp32-noise swaps, each checked by check_parity
    ix.status()
    ix.release()


def test_cross_checks_with_existing_entry_points(knn_lib):
    rows, mu = _mixture(8000, 96, 20, 11)
    rows[100:110] = rows[50]                          # exact ties inside one query's candidates
    assign = np.argmin(((rows[:, None, :] - mu[None]) ** 2).sum(-1), 1).astype(np.int32)
    ix = _index(rows, "cosine")
    ix.set_clusters(mu, assign)
    q = rows[[50, 7, 900, 4000]] + 0.01
    gi, gs, probes = ix.search_clusters(q, 20, 3, return_probes=True)
    for i in range(4):
        cand = _candidates(assign, probes[i])
        keep = np.zeros(len(rows), bool)
        keep[cand] = True
        ix.set_row_mask(keep)                         # nk_search with a row mask equal to the candidate set
        si, ss = ix.search(q[i], 20)
        assert set(si[0].tolist()) == set(gi[i].tolist())
        ix.set_row_mask(None)
        ui, us = ix.score_subset(q[i], cand, 20)      # the previous mirror path, ties in the same order
        assert (ui == gi[i]).all() and (us == gs[i]).all()
    ix.set_clusters(mu, assign)
    ai, _ = ix.search_clusters(q, 20, 20)             # n_probe = K, every row assigned: plain nk_search
    pi, _ = ix.search(q, 20)
    for i in range(4):
        assert set(ai[i].tolist()) == set(pi[i].tolist())
    ix.release()


def test_adversarial_cluster_shapes(knn_lib):
    n, d, K = 40_000, 64, 64
    rows, mu = _mixture(n, d, K, 21)
    assign = np.random.default_rng(1).integers(1, K - 10, n).astype(np.int32)
    assign[: n // 2] = 0                              # one hot cluster with half the rows
    assign[n // 2: n // 2 + 5] = K - 5                # one-row clusters
    assign[n // 2 + 1] = K - 4
    assign[n // 2 + 2] = K - 3
    assign[n // 2 + 10: n // 2 + 200] = -1            # rows in no cluster; clusters K-10 .. K-6 stay empty
    rows[n // 2 + 300] = rows[n // 2 + 301]           # identical rows in different clusters: probe-rank tie order
    assign[n // 2 + 300], assign[n // 2 + 301] = 1, 2
    rows[7] = np.nan                                  # NaN / Inf rows inside the hot cluster
    rows[9, 3] = np.inf
    ix = _index(rows, "cosine")
    ix.set_clusters(mu, assign)
    q = np.repeat(mu[:1], 1024, 0) + np.random.default_rng(3).standard_normal((1024, d)).astype(np.float32) * 0.01
    gi, gs, probes = ix.search_clusters(q, 10, 3, return_probes=True)
    assert (probes[:, 0] == 0).all()                  # the hot cluster is probed by all 1024 queries
    fin = np.isfinite(rows).all(1)
    oi, os_ = _oracle(np.where(fin[:, None], rows, 0), mu, np.where(fin, assign, -1), q, 10, 3, "cosine")
    _compare(rows, q, "cosine", gi, gs, oi, os_)
    # empty / one-row clusters: fewer candidates than k -> sentinel padding
    for P in (1, 4, 10):
        ge, se, pe = ix.search_clusters(mu[K - 5:K - 4], 16, P, return_probes=True)
        cand = _candidates(assign, pe[0])
        assert P > 1 or len(cand) == 3
        assert (ge[0, len(cand):] == SENT).all() and (se[0, len(cand):] == 0).all()
        assert set(ge[0, :min(16, len(cand))].tolist()) <= set(cand.tolist())
    # identical rows, clusters 1 and 2: the one in the cluster probed first comes first
    qt = rows[n // 2 + 300: n // 2 + 301]
    gt, st, pt = ix.search_clusters(qt, 2, K, return_probes=True)
    first = n // 2 + 300 if list(pt[0]).index(1) < list(pt[0]).index(2) else n // 2 + 301
    assert gt[0, 0] == first and st[0, 0] == st[0, 1]
    # NaN / Inf rows score -inf and come last, like the CUDA-core path of nk_search
    few = _index(rows[:12], "dot")
    few.set_clusters(mu[:1], np.zeros(12, np.int32))
    gf, sf = few.search_clusters(mu[:1], 12, 1)
    assert np.isneginf(sf[0, list(gf[0]).index(7)])
    few.set_path("simt")
    pf, psf = few.search(mu[:1], 12)
    assert (pf[0] == gf[0]).all() and np.array_equal(psf[0], sf[0])
    ix.status(); few.release(); ix.release()


def test_row_mask_and_score_floor(knn_lib):
    rows, mu = _mixture(6000, 48, 16, 31)
    assign = np.argmin(((rows[:, None, :] - mu[None]) ** 2).sum(-1), 1).astype(np.int32)
    q = rows[:33] + 0.02
    for metric, floor in (("cosine", 0.9), ("dot", 2.0), ("euclidean", 1.5)):
        ix = _index(rows, metric)
        ix.set_clusters(mu, assign)
        keep = np.random.default_rng(0).random(len(rows)) < 0.5
        ix.set_row_mask(keep)
        ix.set_min_score(floor)
        gi, gs = ix.search_clusters(q, 50, 3)
        oi, os_ = _oracle(rows, mu, assign, q, 50, 3, metric, mask=keep, floor=floor)
        _compare(rows, q, metric, gi, gs, oi, os_)
        ix.set_min_score(1e9 if metric != "euclidean" else 0.0)  # a floor that admits nothing
        gi, gs = ix.search_clusters(q, 50, 3)
        assert (gi == SENT).all() and (gs == 0).all()
        ix.release()


def test_lifecycle(knn_lib):
    from nornicdb_b200.knn import KnnError
    rows, mu = _mixture(2000, 32, 8, 41)
    assign = np.argmin(((rows[:, None, :] - mu[None]) ** 2).sum(-1), 1).astype(np.int32)
    ix = _index(rows, "dot")
    with pytest.raises(KnnError, match="no clusters set"):
        ix.search_clusters(rows[:2], 5, 2)
    ix.set_clusters(mu, assign)
    ix.update_row(5, rows[5] * 100)                  # update_row keeps the clustering and scores the new contents
    gi, gs = ix.search_clusters(rows[5:6], 1, 1)
    assert gi[0, 0] == 5 and abs(gs[0, 0] - float(rows[5].astype(np.float64) @ (rows[5] * 100))) < 1e-3 * abs(gs[0, 0])
    ix.set_clusters(mu, np.full(2000, 3, np.int32))  # re-installing replaces the old clustering
    gi, _, p = ix.search_clusters(mu, 5, 1, return_probes=True)
    for i in range(8):
        assert (gi[i] != SENT).all() if p[i, 0] == 3 else (gi[i] == SENT).all()
    ix.append(rows[:3])
    with pytest.raises(KnnError, match="no clusters set"):
        ix.search_clusters(rows[:2], 5, 2)
    ix.set_clusters(mu, np.append(assign, [0, 0, 0]).astype(np.int32))
    ix.remove_swap(0)
    with pytest.raises(KnnError, match="no clusters set"):
        ix.search_clusters(rows[:2], 5, 2)
    with pytest.raises(KnnError):
        ix.set_clusters(mu, assign)                  # one assignment per row
    ix.set_clusters(mu, np.zeros(len(ix), np.int32))
    with pytest.raises(KnnError):
        ix.search_clusters(rows[:2], 1025, 2)        # k > NK_MAX_K
    with pytest.raises(KnnError):
        ix.search_clusters(rows[:2], 5, 0)           # n_probe = 0
    with pytest.raises(KnnError):
        ix.set_clusters(np.zeros((4097, 32), np.float32), np.zeros(len(ix), np.int32))
    assert ix.search_clusters(rows[:2], 0, 2)[0].shape == (2, 0)
    ix.release()


def test_device_resident_form(knn_lib):
    import torch
    rows, mu = _mixture(20_000, 128, 64, 51)
    assign = np.argmin(((rows[:, None, :] - mu[None]) ** 2).sum(-1), 1).astype(np.int32)
    ix = _index(rows, "cosine")
    ix.set_clusters(mu, assign)
    batches = [rows[np.random.default_rng(s).integers(0, 20_000, Q)] + 0.01 for s, Q in ((1, 64), (2, 1), (3, 300))]
    want = [ix.search_clusters(b, 10, 3, return_probes=True) for b in batches]
    st = torch.cuda.Stream()
    outs = []
    with torch.cuda.stream(st):
        for b in batches:                             # queued back to back, no sync in between
            qd = torch.from_numpy(b).cuda()
            oi = torch.empty((len(b), 10), dtype=torch.int32, device="cuda")
            os_ = torch.empty((len(b), 10), dtype=torch.float32, device="cuda")
            op = torch.empty((len(b), 3), dtype=torch.int32, device="cuda")
            assert ix.search_clusters_device(qd.data_ptr(), len(b), 10, 3, oi.data_ptr(), os_.data_ptr(), op.data_ptr(), st.cuda_stream) == 10
            outs.append((qd, oi, os_, op))
    ix.status(st.cuda_stream)
    for (wi, ws, wp), (_, oi, os_, op) in zip(want, outs):
        assert (oi.cpu().numpy().view(np.uint32) == wi).all()
        assert (os_.cpu().numpy() == ws).all()
        assert (op.cpu().numpy() == wp).all()
    ix.release()


def test_at_scale(knn_lib):
    """N = 2M, d = 1024 mixture (1000 centres, sigma 0.1) held in a torch tensor the index reads in place; K = 1000 from
    device Lloyd passes; Q = 1024, n_probe = 3, k = 10 against a torch fp64 brute force over each query's candidates."""
    import torch
    from nornicdb_b200.knn import KnnIndex
    n, d, K, Q = 2_000_000, 1024, 1000, 1024
    g = torch.Generator(device="cuda").manual_seed(0)
    centres = torch.rand((K, d), generator=g, device="cuda") * 2 - 1
    X = centres[torch.randint(0, K, (n,), generator=g, device="cuda")]
    X += torch.randn((n, d), generator=g, device="cuda") * 0.1
    ix = KnnIndex(d, metric="cosine")
    ix.attach_device_rows(X.data_ptr(), n)
    ix.refresh_shadow()
    rng = np.random.default_rng(0)
    cen = X[torch.from_numpy(rng.choice(n, K, replace=False)).cuda()].cpu().numpy()
    assign = np.zeros(n, np.int32)
    for _ in range(3):
        ix.assign_nearest(cen, assign)
        cen, _ = ix.cluster_means(assign, cen)
    ix.set_clusters(cen, assign)
    q = (X[torch.from_numpy(rng.choice(n, Q, replace=False)).cuda()] + torch.randn((Q, d), generator=g, device="cuda") * 0.05).cpu().numpy()
    gi, gs, probes = ix.search_clusters(q, 10, 3, return_probes=True)
    _check_probes(cen, q, probes)
    order = np.argsort(assign, kind="stable")
    bounds = np.searchsorted(assign[order], np.arange(K + 1))
    qd = torch.from_numpy(q).cuda().double()
    swaps = 0
    for i in range(Q):
        cand = np.concatenate([order[bounds[c]:bounds[c + 1]] for c in probes[i]])
        xs = X[torch.from_numpy(cand).cuda()].double()
        s = ((xs @ qd[i]) / (xs.norm(dim=1) * qd[i].norm())).cpu().numpy()
        o = np.lexsort((np.arange(len(cand)), -s))[:10]
        if not (gi[i] == cand[o]).all():
            pos = {int(r): j for j, r in enumerate(cand)}
            got = s[[pos[int(r)] for r in gi[i]]]
            assert np.abs(got - s[o]).max() <= 2e-6, (i, gi[i], cand[o])
            swaps += 1
        assert np.allclose(gs[i], s[o], rtol=1e-4, atol=1e-6)
    assert swaps <= Q // 100
    ix.status()
    ix.release()
    del X
