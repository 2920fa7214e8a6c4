"""The device-resident (asynchronous) search API on adversarial data, the CTA-pair kernel at every prune width, and the
documented environment switches.

nk_search_device / nk_search_keys_device / nk_search_sharded_device queue the whole filter tail up front: a first-stage
overflow skips the TF32 retry stage and goes straight to the exact twin (3xTF32 for cosine / dot over fp32 rows, the
CUDA-core scan otherwise), whose merge overwrites the caller's buffers.  Every adversarial test here says which stage
answered, through the cumulative counters (exact_stage_runs, bf16_stage_retries): a stage that overflows has its own
answer thrown away, so a test of a first-stage kernel must show that it did not overflow, and a test of the tail must
show that the tail ran exactly once per search."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest

from parity import check_parity, torch_fp64_topk

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METRICS = ["cosine", "dot", "euclidean"]


# ---- helpers ---------------------------------------------------------------------------------------------------------
def _counters(ix):
    c = ix.debug_counters()
    return np.array([c["exact_stage_runs"], c["bf16_stage_retries"]])


def _launch(ix, qd, Q, k, stream, keys=False):
    """Queue one device-resident search on `stream`; returns its output tensors (nothing is synchronised)."""
    import torch
    with torch.cuda.stream(stream):
        if keys:
            out = (torch.empty((Q, k), dtype=torch.int64, device="cuda"),)
            assert ix.search_keys_device(qd.data_ptr(), Q, k, out[0].data_ptr(), stream.cuda_stream) == k
        else:
            out = (torch.empty((Q, k), dtype=torch.int32, device="cuda"), torch.empty((Q, k), dtype=torch.float32, device="cuda"))
            assert ix.search_device(qd.data_ptr(), Q, k, out[0].data_ptr(), out[1].data_ptr(), stream.cuda_stream) == k
    return out


def _to_numpy(out):
    if len(out) == 1:
        return out[0].cpu().numpy()
    return out[0].cpu().numpy().view(np.uint32), out[1].cpu().numpy()


def _upload_queries(q, stream):
    import torch
    with torch.cuda.stream(stream):
        return torch.from_numpy(np.ascontiguousarray(q, dtype=np.float32)).cuda()


def device_search(ix, q, k, keys=False):
    """search_device (or search_keys_device) on an explicit non-default stream: handle 0 would mean "the index's own
    stream" to the C ABI.  Synchronises only that stream, then asks the index for its status word."""
    import torch
    st = torch.cuda.Stream()
    qd = _upload_queries(q, st)
    out = _launch(ix, qd, q.shape[0], k, st, keys=keys)
    st.synchronize()
    res = _to_numpy(out)
    ix.status(st.cuda_stream)
    return res


def merge_keys(keys, metric):
    """The library's own key decode: nk_merge_keys_device over [lists, Q, k] keys."""
    import torch
    from nornicdb_b200.knn import merge_keys_device
    keys = np.ascontiguousarray(keys.reshape((-1,) + keys.shape[-2:]))
    L, Q, k = keys.shape
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        kd = torch.from_numpy(keys).cuda()
        oi = torch.empty((Q, k), dtype=torch.int32, device="cuda")
        os_ = torch.empty((Q, k), dtype=torch.float32, device="cuda")
        merge_keys_device(0, kd.data_ptr(), L, Q, k, metric, oi.data_ptr(), os_.data_ptr(), st.cuda_stream)
    st.synchronize()
    return oi.cpu().numpy().view(np.uint32), os_.cpu().numpy()


def _same_row_scores(a_idx, a_sc, b_idx, b_sc, rtol=2e-6):
    """Rows returned by both results carry the same score to `rtol` relative."""
    for qi in range(a_idx.shape[0]):
        sa = dict(zip(a_idx[qi].tolist(), a_sc[qi].tolist()))
        for r, s in zip(b_idx[qi].tolist(), b_sc[qi].tolist()):
            if r in sa:
                assert abs(sa[r] - s) <= rtol * max(abs(s), 1e-3), (qi, r, sa[r], s)


def _anti_aligned(oracle, Q, d, base, seed):
    """Uniform queries pointing away from `base`: the near-duplicate clump around `base` ranks last for every metric, so
    these batches see the clump as far-away rows (no near-ties) while sharing the index with the adversarial batches."""
    q = oracle.fill_uniform(Q, d, seed).astype(np.float64)
    u = base / np.linalg.norm(base)
    q -= np.outer(q @ u, u)
    q -= 0.5 * np.linalg.norm(q, axis=1, keepdims=True) * u[None, :]
    return np.ascontiguousarray(q, dtype=np.float32)


def near_dup_corpus(oracle, kind, Q):
    """The adversarial corpora of the overflow tests: (rows to upload, their exact fp32 values, queries, dtype, path, base).
      filter : 20k fp32 copies of one vector + 1e-5 noise (every seventh row uniform): overflows the TF32 filter's k_emit
      shadow : 160k copies + 1e-4 noise: > 768 rows per CTA inside the 16-bit margin, more than one buffer holds
      f16/bf16 : the shadow construction stored in 16 bits (noise sized to the format's ulp, so that rows differ in a few
                 last bits): the 16-bit kernel runs in place and the CUDA-core scan is the exact twin
    Queries are the base vector + 1e-3 noise."""
    from nornicdb_b200.knn import from_bf16_bits, to_bf16_bits
    n, seed, noise = {"filter": (20_000, 0, 1e-5), "shadow": (160_000, 1, 1e-4), "f16": (160_000, 2, 1e-4),
                      "bf16": (160_000, 3, 1e-3)}[kind]
    d = 128
    rng = np.random.default_rng(seed)
    base = oracle.fill_uniform(1, d, 9)[0]
    rows = np.tile(base, (n, 1)) + rng.standard_normal((n, d)).astype(np.float32) * np.float32(noise)
    rows[::7] = oracle.fill_uniform(len(rows[::7]), d, 10)
    q = (base[None, :] + rng.standard_normal((Q, d)).astype(np.float32) * 1e-3).astype(np.float32)
    if kind == "f16":
        up = rows.astype(np.float16)
        return up, up.astype(np.float32), q, "f16", "shadow", base
    if kind == "bf16":
        up = to_bf16_bits(rows)
        return up, from_bf16_bits(up), q, "bf16", "shadow", base
    return rows, rows, q, "f32", kind, base


def gpu_reference(rows, q, k, metric):
    """fp64 brute force with torch on the GPU (for the large batches; ties are rare on these corpora)."""
    import torch
    x = torch.from_numpy(np.ascontiguousarray(rows, dtype=np.float32)).cuda()
    return torch_fp64_topk(x.shape[0], x.shape[1], q, k, metric, x.shape[0], lambda lo, cnt: x[lo:lo + cnt])


def _index(rows, metric, dtype="f32", path="auto", row_base=0):
    from nornicdb_b200.knn import KnnIndex
    ix = KnnIndex(rows.shape[1], metric=metric, dtype=dtype)
    if row_base:
        ix.set_row_base(row_base)
    ix.upload(rows)
    ix.set_path(path)
    return ix


# ---- A1. overflow through the device API -----------------------------------------------------------------------------
@pytest.mark.parametrize("Q", [40, 130])
@pytest.mark.parametrize("kind", ["filter", "shadow", "f16", "bf16"])
@pytest.mark.parametrize("metric", METRICS)
def test_device_search_overflow_takes_the_exact_stage(knn_lib, oracle_mod, metric, kind, Q):
    """Near-duplicates overflow the first stage; the asynchronous tail goes straight to the exact twin (3xTF32 for cosine /
    dot over fp32 rows, the CUDA-core scan for euclidean and 16-bit rows), which must answer like the fp64 oracle.  At
    Q = 130 the 3xTF32 twin takes three 64-query passes."""
    k = 10
    up, exact, q, dtype, path, _ = near_dup_corpus(oracle_mod, kind, Q)
    oi, os_ = oracle_mod.knn_exact64(exact, q, k, metric)
    ix = _index(up, metric, dtype, path)
    c0 = _counters(ix)
    gi, gs = device_search(ix, q, k)
    c1 = _counters(ix)
    assert ix.last_path() == path
    assert (c1 - c0).tolist() == [1, 0], (c1 - c0)  # exactly one exact-stage run, no TF32 retry on the asynchronous path
    check_parity(exact, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)
    # the host-synchronous API on the same input (its tail usually answers from the TF32 retry stage)
    si, ss = ix.search(q, k)
    assert ix.debug_flags()[0] == 0
    ix.release()
    check_parity(exact, q, k, metric, si, ss, oi, os_, swap_eps=5e-6)
    _same_row_scores(gi, gs, si, ss)


@pytest.mark.parametrize("Q", [40, 130])
@pytest.mark.parametrize("path", ["filter", "shadow"])
@pytest.mark.parametrize("metric", METRICS)
def test_device_search_k_or_more_nan_rows(knn_lib, oracle_mod, metric, path, Q):
    """k or more NaN rows in one tile (test_gpu_round2's construction at Q = 40 / 130).  Every prune and the finish step
    take the k-th FINITE bound (NaN rows are kept aside as undecidable), so this is expected NOT to overflow: the first
    stage answers, and it must rank the NaN rows last."""
    n, d, k = 5000, 64, 5
    rows = oracle_mod.fill_uniform(n, d, 31)
    q = oracle_mod.fill_uniform(Q, d, 32)
    bad = np.arange(100, 120)
    rows[bad, 3] = np.nan
    good = np.setdiff1d(np.arange(n), bad)
    ix = _index(rows, metric, path=path)
    c0 = _counters(ix)
    gi, gs = device_search(ix, q, k)
    c1 = _counters(ix)
    si, ss = ix.search(q, k)
    ix.release()
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)
    oi, os_ = oracle_mod.knn_exact64(rows[good], q, k, metric)
    check_parity(rows, q, k, metric, gi, gs, good[oi], os_)
    assert (gi == si).all() and (gs.view(np.uint32) == ss.view(np.uint32)).all()


# ---- A2. keys output, single list and two half shards ----------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_keys_device_overflow_single_list_and_half_shards(knn_lib, oracle_mod, metric):
    """search_keys_device on an overflowing shard, decoded by merge_keys_device; then two half shards of which only the
    first holds the near-duplicate block (it answers from the exact twin, the other from the filter) merged into one
    result — the mix nk_search_sharded_device produces."""
    k, Q = 10, 40
    rows, _, q, _, _, _ = near_dup_corpus(oracle_mod, "filter", Q)
    n, d = rows.shape
    h = n // 2
    rows[h:] = oracle_mod.fill_uniform(n - h, d, 12)  # the second half: uniform rows only
    oi, os_ = oracle_mod.knn_exact64(rows, q, k, metric)
    full = _index(rows, metric, path="filter")
    c0 = _counters(full)
    keys = device_search(full, q, k, keys=True)
    c1 = _counters(full)
    di, ds = device_search(full, q, k)
    c2 = _counters(full)
    full.release()
    assert (c1 - c0).tolist() == [1, 0] and (c2 - c1).tolist() == [1, 0], (c0, c1, c2)
    ki, ks = merge_keys(keys, metric)
    check_parity(rows, q, k, metric, ki, ks, oi, os_, swap_eps=5e-6)
    assert (ki == di).all() and (ks.view(np.uint32) == ds.view(np.uint32)).all()  # one decode, same bits
    halves, deltas, parts = [], [], []
    for g, (lo, hi) in enumerate([(0, h), (h, n)]):
        ix = _index(rows[lo:hi], metric, path="filter", row_base=lo)
        c0 = _counters(ix)
        parts.append(device_search(ix, q, k, keys=True))
        deltas.append((_counters(ix) - c0).tolist())
        ix.release()
    assert deltas == [[1, 0], [0, 0]], deltas
    mi, ms = merge_keys(np.stack(parts), metric)
    check_parity(rows, q, k, metric, mi, ms, oi, os_, swap_eps=5e-6)
    _same_row_scores(di, ds, mi, ms)


# ---- A3. row mask and score floor on the tail -------------------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_device_tail_honours_row_mask_and_score_floor(knn_lib, oracle_mod, metric):
    """One batch: 20 queries on the near-duplicate block (they make the whole search overflow, so the exact twin re-runs
    every query) and 20 uniform queries whose lists the floor cuts half way.  The exact stage must honour the mask and
    the floor; unused slots read 0xFFFFFFFF."""
    k = 20
    rows, _, qa, _, _, _ = near_dup_corpus(oracle_mod, "filter", 20)
    n, d = rows.shape
    q = np.concatenate([qa, oracle_mod.fill_uniform(20, d, 13)])
    keep = np.random.default_rng(14).random(n) < 0.8
    sub = np.where(keep)[0]
    oi, os_ = oracle_mod.knn_exact64(rows[sub], q, k, metric)
    oi = sub[oi]
    floor = float(np.median(os_[20:, k // 2]))
    near = os_[:20] <= floor if metric == "euclidean" else os_[:20] >= floor
    assert near.all()  # the floor cuts only the uniform queries' lists
    ix = _index(rows, metric, path="filter")
    ix.set_row_mask(keep)
    ix.set_min_score(floor)
    c0 = _counters(ix)
    gi, gs = device_search(ix, q, k)
    c1 = _counters(ix)
    ix.release()
    assert (c1 - c0).tolist() == [1, 0], (c1 - c0)
    for qi in range(q.shape[0]):
        ok = os_[qi] <= floor if metric == "euclidean" else os_[qi] >= floor
        noise = np.abs(os_[qi] - floor) <= 2e-6 * max(1.0, abs(floor))  # within fp32 noise of the floor: either side
        got = gi[qi][gi[qi] != 0xFFFFFFFF]
        assert keep[got.astype(np.int64)].all()
        assert (gi[qi][len(got):] == 0xFFFFFFFF).all()
        if qi < 20:  # near-duplicate queries: a full list; near-ties inside 3xTF32 noise may swap (check_parity below)
            assert len(got) == k, (qi, got)
        else:        # uniform queries: exactly the kept rows above the floor
            assert set(oi[qi][ok & ~noise].tolist()) <= set(got.tolist()) <= set(oi[qi][ok | noise].tolist()), (qi, got)
        m = len(got)
        check_parity(rows, q[qi:qi + 1], m, metric, gi[qi:qi + 1, :m], gs[qi:qi + 1, :m], oi[qi:qi + 1, :m], os_[qi:qi + 1, :m],
                     swap_eps=5e-6)


# ---- A4. back-to-back pipeline, no host synchronisation ---------------------------------------------------------------
@pytest.mark.parametrize("metric", ["cosine", "euclidean"])
def test_pipeline_of_device_searches_without_host_sync(knn_lib, oracle_mod, metric):
    """Six searches queued back to back on one index and one stream: uniform batches (16-bit filter; CTA pairs at
    Q = 300), two near-duplicate batches (overflow -> exact twin), a Q = 3 CUDA-core search and a k = 1500 search (bounded
    CUDA-core passes + key decode).  Catches state one search leaks into the next: the status words the prep kernel
    clears, the finish-CTA counter, the shared gtau / gcount words."""
    import torch
    up, rows, qa, _, _, base = near_dup_corpus(oracle_mod, "shadow", 130)
    d = rows.shape[1]
    batches = [  # (queries, k, path, overflows)
        (_anti_aligned(oracle_mod, 64, d, base, 20), 10, "auto", False),
        (qa[:40], 10, "auto", True),
        (_anti_aligned(oracle_mod, 3, d, base, 21), 10, "simt", False),
        (_anti_aligned(oracle_mod, 300, d, base, 22), 10, "auto", False),
        (qa, 10, "auto", True),
        (_anti_aligned(oracle_mod, 8, d, base, 23), 1500, "auto", False),
    ]
    ix = _index(up, metric)
    st = torch.cuda.Stream()
    qds = [_upload_queries(b[0], st) for b in batches]
    c0 = _counters(ix)
    outs = []
    for (q, k, path, _), qd in zip(batches, qds):
        ix.set_path(path)  # host-side state, read when the search is queued
        outs.append(_launch(ix, qd, q.shape[0], k, st))
    st.synchronize()
    res = [_to_numpy(o) for o in outs]
    ix.status(st.cuda_stream)
    c1 = _counters(ix)
    assert (c1 - c0).tolist() == [sum(b[3] for b in batches), 0], (c1 - c0)
    for (q, k, path, ovf), (gi, gs) in zip(batches, res):
        oi, os_ = oracle_mod.knn_exact64(rows, q, k, metric)
        check_parity(rows, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)
        ix.set_path(path)
        c0 = _counters(ix)
        ai, as_ = device_search(ix, q, k)
        assert (_counters(ix) - c0).tolist() == [int(ovf), 0], (q.shape, k, ovf)
        if not ovf:  # the same batch searched alone: the same bits
            assert (ai == gi).all() and (as_.view(np.uint32) == gs.view(np.uint32)).all(), (q.shape, k)
    ix.release()


# ---- A5. a host-synchronous retry, then a device search ---------------------------------------------------------------
@pytest.mark.parametrize("metric", METRICS)
def test_sync_retry_then_device_search(knn_lib, oracle_mod, metric):
    """ix.search on near-duplicates goes through the TF32 retry stage and leaves the retry marker set; the next device
    search (easy queries) must neither re-run a stage nor inherit anything from it."""
    k = 10
    up, rows, qa, _, _, base = near_dup_corpus(oracle_mod, "shadow", 40)
    ix = _index(up, metric, path="shadow")
    c0 = _counters(ix)
    si, ss = ix.search(qa, k)
    c1 = _counters(ix)
    assert c1[1] - c0[1] == 1 and ix.debug_flags()[3] == 1, (c0, c1)
    q = _anti_aligned(oracle_mod, 64, rows.shape[1], base, 30)
    gi, gs = device_search(ix, q, k)
    c2 = _counters(ix)
    fl = ix.debug_flags()
    ix.release()
    assert (c2 - c1).tolist() == [0, 0], (c1, c2)
    assert fl[1] == 0 and fl[3] == 0, fl
    oi, os_ = oracle_mod.knn_exact64(rows, qa, k, metric)
    check_parity(rows, qa, k, metric, si, ss, oi, os_, swap_eps=5e-6)
    oi, os_ = oracle_mod.knn_exact64(rows, q, k, metric)
    check_parity(rows, q, k, metric, gi, gs, oi, os_)


# ---- A6. peer exchange with one rank overflowing ----------------------------------------------------------------------
@pytest.mark.parametrize("metric", ["cosine", "euclidean"])
def test_exchange_two_ranks_one_overflowing(knn_lib, oracle_mod, metric):
    """Two ranks on cuda:0; rank 0's shard holds the near-duplicate block.  Rank 0 answers from the exact twin, rank 1 from
    the filter; both then push, wait and merge: finish -> exact -> merge -> push -> wait/merge on the same stream."""
    import torch
    from nornicdb_b200.knn import Comm
    k, Q, reps = 10, 16, 2
    rows, _, q, _, _, _ = near_dup_corpus(oracle_mod, "filter", Q)
    n, d = rows.shape
    rows = np.concatenate([rows, oracle_mod.fill_uniform(n, d, 15)])
    bounds = [(0, n), (n, 2 * n)]
    ixs, comms, outs = [], [], []
    qd = torch.from_numpy(q).cuda()
    for r, (lo, hi) in enumerate(bounds):
        ixs.append(_index(rows[lo:hi], metric, path="filter", row_base=lo))
        comms.append(Comm(0, r, 2, Q * k * 8))
        outs.append((torch.empty((Q, k), dtype=torch.int32, device="cuda"), torch.empty((Q, k), dtype=torch.float32, device="cuda")))
    Comm.connect_local(comms)
    torch.cuda.synchronize()
    c0 = [_counters(ix) for ix in ixs]
    for _ in range(reps):
        for r in range(2):
            ixs[r].search_sharded_device(comms[r], qd.data_ptr(), Q, k, outs[r][0].data_ptr(), outs[r][1].data_ptr())
        for r in range(2):
            comms[r].status()
            ixs[r].status()
    deltas = [(_counters(ix) - c).tolist() for ix, c in zip(ixs, c0)]
    res = [(o[0].cpu().numpy().view(np.uint32), o[1].cpu().numpy()) for o in outs]
    for r in range(2):
        comms[r].release()
        ixs[r].release()
    assert deltas == [[reps, 0], [0, 0]], deltas
    oi, os_ = oracle_mod.knn_exact64(rows, q, k, metric)
    for gi, gs in res:
        check_parity(rows, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)
    assert (res[0][0] == res[1][0]).all() and (res[0][1].view(np.uint32) == res[1][1].view(np.uint32)).all()


# ---- B7. the CTA-pair kernel at every prune width ---------------------------------------------------------------------
PAIR_N, PAIR_D = 200_000, 128
PAIR_KS = [10, 127, 128, 150, 160, 161, 192]


@pytest.fixture(scope="module")
def pair_corpora(knn_lib, oracle_mod):
    """One 200k x 128 uniform index per metric (>= 8 pair tiles per CTA pair even with a single query group) and the fp64
    top-192 of every query batch, computed once with torch on the GPU."""
    import torch
    from nornicdb_b200.knn import KnnIndex, fill_uniform_device
    x = torch.empty((PAIR_N, PAIR_D), dtype=torch.float32, device="cuda")
    fill_uniform_device(0, x.data_ptr(), PAIR_N, PAIR_D, 202, 0, 0)
    torch.cuda.synchronize()
    cache = {"rows": x, "host": x.cpu().numpy(), "ix": {}, "ref": {}}

    def get(metric, Q):
        if metric not in cache["ix"]:
            ix = KnnIndex(PAIR_D, metric=metric)
            ix.fill_uniform(PAIR_N, 202)  # the same counter-based generator as fill_uniform_device
            ix.set_path("shadow")
            cache["ix"][metric] = ix
        q = oracle_mod.fill_uniform(Q, PAIR_D, 203 + Q)
        if (metric, Q) not in cache["ref"]:
            cache["ref"][(metric, Q)] = torch_fp64_topk(PAIR_N, PAIR_D, q, max(PAIR_KS), metric, PAIR_N, lambda lo, cnt: x[lo:lo + cnt])
        return cache["ix"][metric], q, cache["host"], cache["ref"][(metric, Q)]

    yield get
    for ix in cache["ix"].values():
        ix.release()


@pytest.mark.parametrize("k", PAIR_KS)
@pytest.mark.parametrize("Q", [256, 520, 1024])
@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_every_prune_width_without_overflow(pair_corpora, metric, Q, k):
    """Uniform data, so nothing may overflow: the pair kernel's own answer is what is checked.  The first in-loop prune sees
    512 keys (k <= 127, warp_prune<16>), 640 (k = 128..159, warp_prune<22>) or 768 / 896 (k >= 160, the full-width select);
    Q = 520 adds a single-CTA remainder of 8 queries, Q = 1024 runs four query groups."""
    ix, q, host, (ri, rs) = pair_corpora(metric, Q)
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    fl = ix.debug_flags()
    assert ix.last_path() == "shadow"
    assert fl[0] == 0 and fl[3] == 0, fl
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)  # no retry, no exact stage
    swaps = check_parity(host, q, k, metric, gi, gs, ri[:, :k], rs[:, :k])
    assert swaps <= Q * k // 2000, swaps


# ---- B8. near-ties at Q >= 256 ----------------------------------------------------------------------------------------
def _clustered(n, d, seed):
    from nornicdb_b200.knn import KnnIndex
    ix = KnnIndex(d, metric="cosine")
    ix.fill_clustered(n, seed, n_centres=40, sigma=0.1)
    rows = ix.read_rows(0, n)
    ix.release()
    return rows


@pytest.mark.parametrize("Q", [300, 1024])
@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_clustered_corpus(knn_lib, oracle_mod, metric, Q):
    """Gaussian mixture (40 centres, sigma 0.1), queries = members + noise: near-ties everywhere.  Expected NOT to
    overflow (none of the six cases does on a B200): the in-loop prunes must keep every row inside the 16-bit margin.
    Q = 300 is one pair launch plus a 44-query single-CTA remainder."""
    n, d, k = 200_000, 128, 10
    rows = _clustered(n, d, 4343)
    rng = np.random.default_rng(40)
    q = (rows[rng.integers(0, n, Q)] + rng.standard_normal((Q, d)).astype(np.float32) * 0.05).astype(np.float32)
    ix = _index(rows, metric, path="shadow")
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    ix.release()
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)
    oi, os_ = gpu_reference(rows, q, k, metric)
    check_parity(rows, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)


@pytest.mark.parametrize("Q", [300, 1024])
@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_mild_near_duplicates(knn_lib, oracle_mod, metric, Q):
    """9000 near-copies of one vector (noise 2e-3) among 200k uniform rows, half of the queries on them: about 60 copies
    per CTA, all close to the k-th bound.  The in-loop prunes must keep them and the finish step re-score them.  Expected
    NOT to overflow."""
    n, d, k = 200_000, 64, 10
    rng = np.random.default_rng(41)
    base = oracle_mod.fill_uniform(1, d, 9)[0]
    rows = oracle_mod.fill_uniform(n, d, 42)
    dup = rng.choice(n, 9000, replace=False)
    rows[dup] = base[None, :] + rng.standard_normal((9000, d)).astype(np.float32) * 2e-3
    q = oracle_mod.fill_uniform(Q, d, 43)
    q[: Q // 2] = base[None, :] + rng.standard_normal((Q // 2, d)).astype(np.float32) * 1e-3
    ix = _index(rows, metric, path="shadow")
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    ix.release()
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)
    oi, os_ = gpu_reference(rows, q, k, metric)
    check_parity(rows, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)


# ---- B9. floor, NaN rows, row mask and 16-bit corpora at Q >= 256 ------------------------------------------------------
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_score_floor_and_row_mask(knn_lib, oracle_mod, metric, masked):
    """test_score_floor_inside_kernels at Q = 300 on path="shadow" (pair kernel + single-CTA remainder), with and without
    a row mask.  Uniform data: no overflow allowed."""
    n, d, Q, k = 60_000, 128, 300, 20
    rows = oracle_mod.fill_uniform(n, d, 8)
    q = oracle_mod.fill_uniform(Q, d, 9)
    keep = np.random.default_rng(50).random(n) < 0.6 if masked else np.ones(n, dtype=bool)
    sub = np.where(keep)[0]
    oi, os_ = oracle_mod.knn_exact64(rows[sub], q, k, metric)
    oi = sub[oi]
    floor = float(np.median(os_[:, k // 2]))
    ix = _index(rows, metric, path="shadow")
    if masked:
        ix.set_row_mask(keep)
    ix.set_min_score(floor)
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    ix.release()
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)
    for qi in range(Q):
        ok = os_[qi] <= floor if metric == "euclidean" else os_[qi] >= floor
        noise = np.abs(os_[qi] - floor) <= 2e-6 * max(1.0, abs(floor))
        got = gi[qi][gi[qi] != 0xFFFFFFFF]
        assert set(oi[qi][ok & ~noise].tolist()) <= set(got.tolist()) <= set(oi[qi][ok | noise].tolist()), (qi, got)
        assert (gi[qi][len(got):] == 0xFFFFFFFF).all()
        assert np.allclose(gs[qi][:len(got)], os_[qi][:len(got)], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_nan_and_inf_rows(knn_lib, oracle_mod, metric):
    """test_nan_and_inf_rows_on_every_path at Q = 300 on path="shadow": NaN / Inf rows rank last, the others unaffected."""
    n, d, Q, k = 60_000, 64, 300, 10
    rows = oracle_mod.fill_uniform(n, d, 21)
    q = oracle_mod.fill_uniform(Q, d, 22)
    bad = np.array([0, 17, 255, 256, 3000, 59_999])
    rows[bad[:4], 5] = np.nan
    rows[bad[4:], 7] = np.inf if metric != "dot" else np.nan  # dot with +inf would legitimately rank first
    good = np.setdiff1d(np.arange(n), bad)
    ix = _index(rows, metric, path="shadow")
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    fl = ix.debug_flags()
    ix.release()
    assert fl[0] == 0 and (c1 - c0).tolist() == [0, 0], (fl, c1 - c0)
    oi, os_ = oracle_mod.knn_exact64(rows[good], q, k, metric)
    check_parity(rows, q, k, metric, gi, gs, good[oi], os_)


@pytest.mark.parametrize("k", [10, 150])
@pytest.mark.parametrize("dtype", ["f16", "bf16"])
@pytest.mark.parametrize("metric", METRICS)
def test_pair_kernel_16bit_corpora(knn_lib, oracle_mod, metric, dtype, k):
    """fp16 / bf16 corpora scanned in place on CTA pairs at Q = 512 (two query groups).  No overflow allowed."""
    from nornicdb_b200.knn import KnnIndex, from_bf16_bits, to_bf16_bits
    n, d, Q = 120_000, 128, 512
    f32 = oracle_mod.fill_uniform(n, d, 61)
    up = f32.astype(np.float16) if dtype == "f16" else to_bf16_bits(f32)
    exact = up.astype(np.float32) if dtype == "f16" else from_bf16_bits(up)
    q = oracle_mod.fill_uniform(Q, d, 62)
    ix = KnnIndex(d, metric=metric, dtype=dtype)
    ix.upload(up)
    ix.set_path("shadow")
    c0 = _counters(ix)
    gi, gs = ix.search(q, k)
    c1 = _counters(ix)
    ix.release()
    assert (c1 - c0).tolist() == [0, 0], (c1 - c0)
    oi, os_ = gpu_reference(exact, q, k, metric)
    swaps = check_parity(exact, q, k, metric, gi, gs, oi, os_)
    assert swaps <= Q * k // 2000, swaps


# ---- C10. the documented environment switches give the same answers ----------------------------------------------------
SWITCHES = [None, {"NK_PDL": "0"}, {"NK_SHADOW": "0"}, {"NK_TAU_SAMPLE": "0"}, {"NK_PRUNE_TRIGGER": "-1"},
            {"NK_TC_QGROUPS": "1"}, {"NK_TC_QGROUPS": "2"}, {"NK_PAIR": "0"}, {"NK_PAIR_GROUPS": "1"}, {"NK_PAIR_GROUPS": "2"}]
SWITCH_N, SWITCH_D = 100_000, 128
# (name, corpus, metric, Q, k)
BATTERY = [(f"uniform_q{Q}_k{k}", "uniform", "cosine", Q, k) for Q in (64, 300, 1024) for k in (10, 150)] + [
    ("clustered_q64", "clustered", "euclidean", 64, 10), ("f16_q64", "f16", "dot", 64, 10)]

CHILD = textwrap.dedent("""
    import sys
    import numpy as np
    import torch
    sys.path.insert(0, sys.argv[1])
    sys.path.insert(0, sys.argv[1] + "/tests")
    import oracle
    from nornicdb_b200.knn import KnnIndex
    from test_gpu_async_tail import BATTERY, SWITCH_N, SWITCH_D, switch_queries, _counters, device_search
    out = {}
    for name, corpus, metric, Q, k in BATTERY:
        ix = KnnIndex(SWITCH_D, metric=metric, dtype="f16" if corpus == "f16" else "f32")
        if corpus == "clustered":
            ix.fill_clustered(SWITCH_N, 505, n_centres=40, sigma=0.1)
        else:
            ix.fill_uniform(SWITCH_N, 504)
        q = switch_queries(oracle, corpus, Q)
        for api in ("search", "device"):
            c0 = _counters(ix)
            gi, gs = ix.search(q, k) if api == "search" else device_search(ix, q, k)
            c1 = _counters(ix)
            out[f"{name}/{api}/idx"] = gi
            out[f"{name}/{api}/score"] = gs
            out[f"{name}/{api}/counters"] = c1 - c0
            out[f"{name}/{api}/path"] = np.array(ix.last_path())
        out[f"{name}/fatal"] = np.array(ix.debug_flags()[0])
        ix.release()
    np.savez(sys.argv[2], **out)
""")


def switch_queries(oracle, corpus, Q):
    if corpus == "clustered":  # members of the corpus + noise (the corpus comes from the device generator)
        from nornicdb_b200.knn import KnnIndex
        ix = KnnIndex(SWITCH_D, metric="euclidean")
        ix.fill_clustered(SWITCH_N, 505, n_centres=40, sigma=0.1)
        rng = np.random.default_rng(506)
        rows = ix.read_rows(0, SWITCH_N)
        ix.release()
        return (rows[rng.integers(0, SWITCH_N, Q)] + rng.standard_normal((Q, SWITCH_D)).astype(np.float32) * 0.05).astype(np.float32)
    return oracle.fill_uniform(Q, SWITCH_D, 507)


def _switch_run(tmp_path, env_extra):
    tag = "default" if env_extra is None else "_".join(f"{a}{b}" for a, b in env_extra.items())
    path = str(tmp_path / f"{tag}.npz")
    env = {key: v for key, v in os.environ.items() if not key.startswith("NK_")}
    env.update(env_extra or {})
    env["PYTHONDONTWRITEBYTECODE"] = "1"  # the child imports this module from the (possibly read-only) source tree
    r = subprocess.run([sys.executable, "-s", "-c", CHILD, ROOT, path], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (tag, r.stdout[-2000:], r.stderr[-4000:])
    return dict(np.load(path))


@pytest.fixture(scope="module")
def switch_reference(knn_lib, oracle_mod, tmp_path_factory):
    """The default settings' results (child process) and the fp64 oracle of every battery case."""
    import torch
    from nornicdb_b200.knn import KnnIndex
    base = _switch_run(tmp_path_factory.mktemp("switch_default"), None)
    ref = {}
    for name, corpus, metric, Q, k in BATTERY:
        ix = KnnIndex(SWITCH_D, metric=metric, dtype="f16" if corpus == "f16" else "f32")
        if corpus == "clustered":
            ix.fill_clustered(SWITCH_N, 505, n_centres=40, sigma=0.1)
        else:
            ix.fill_uniform(SWITCH_N, 504)
        rows = ix.read_rows(0, SWITCH_N).astype(np.float32)
        ix.release()
        q = switch_queries(oracle_mod, corpus, Q)
        x = torch.from_numpy(rows).cuda()
        oi, os_ = torch_fp64_topk(SWITCH_N, SWITCH_D, q, k, metric, SWITCH_N, lambda lo, cnt: x[lo:lo + cnt])
        ref[name] = (rows, q, metric, k, oi, os_)
        for api in ("search", "device"):
            swaps = check_parity(rows, q, k, metric, base[f"{name}/{api}/idx"], base[f"{name}/{api}/score"], oi, os_, swap_eps=5e-6)
            assert swaps <= Q * k // 2000, (name, api, swaps)
        assert int(base[f"{name}/fatal"]) == 0
    return base, ref


@pytest.mark.parametrize("switch", SWITCHES[1:], ids=lambda s: "_".join(f"{a}={b}" for a, b in s.items()))
def test_environment_switches_give_the_same_answers(switch_reference, tmp_path, switch):
    """Every final score comes from exact fp32 rescoring of a superset of the true top-k, so a search that takes no exact
    stage must return the same bits under every documented switch.  Where either run used the exact stage, the
    switched result must still match the fp64 oracle."""
    base, ref = switch_reference
    got = _switch_run(tmp_path, switch)
    for name, _, _, _, _ in BATTERY:
        rows, q, metric, k, oi, os_ = ref[name]
        assert int(got[f"{name}/fatal"]) == 0, name
        for api in ("search", "device"):
            key = f"{name}/{api}"
            gi, gs = got[key + "/idx"], got[key + "/score"]
            if base[key + "/counters"][0] == 0 and got[key + "/counters"][0] == 0:
                assert (gi == base[key + "/idx"]).all(), key
                if str(got[key + "/path"]) == str(base[key + "/path"]):
                    assert (gs.view(np.uint32) == base[key + "/score"].view(np.uint32)).all(), key
                else:  # (NK_SHADOW=0 moves a 16-bit corpus to the CUDA-core scan: fp32 scores of its own summation order)
                    assert np.allclose(gs, base[key + "/score"], rtol=2e-6, atol=1e-7), key
            else:
                check_parity(rows, q, k, metric, gi, gs, oi, os_, swap_eps=5e-6)
            # (measured on a B200: no setting takes the retry or exact stage on this battery, so every case above is
            # compared bit for bit; a switch that starts overflowing is still held to the oracle)
