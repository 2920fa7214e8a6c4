"""Parity checker: CUDA result vs the fp64 oracle on the same inputs (SURVEY.md §8d "parity rule").

  * scores: within 1e-4 relative of the oracle's fp64 score at the same rank (absolute floor 1e-6);
  * index sets: identical to the oracle's (score desc, row asc) top-k.  Two fp32 summation orders may
    legitimately swap neighbours whose fp64 scores are closer than fp32 noise; such "boundary swaps" are
    accepted only when the fp64 scores of the swapped rows differ by < swap_eps * scale, and are counted.
Returns the number of boundary swaps (0 for almost every case)."""
import numpy as np

REL_TOL = 1e-4   # north_star: "distances within 1e-4 relative for fp32"
ABS_FLOOR = 1e-6


def exact_scores_for(rows, q, idx, metric):
    """fp64 score of the given rows for one query (rows: full corpus array or callable(idx)->rows)."""
    sel = rows(idx) if callable(rows) else rows[idx]
    x = np.asarray(sel, dtype=np.float64)
    qq = np.asarray(q, dtype=np.float64)
    if metric == "dot":
        return x @ qq
    if metric == "cosine":
        den = np.linalg.norm(x, axis=1) * np.linalg.norm(qq)
        with np.errstate(invalid="ignore", divide="ignore"):
            s = np.where(den > 0, (x @ qq) / den, 0.0)
        return s
    return np.sqrt(((x - qq[None, :]) ** 2).sum(1))


def check_parity(rows, queries, k, metric, g_idx, g_score, o_idx, o_score, row_base=0, swap_eps=2e-6):
    queries = np.asarray(queries, dtype=np.float32)
    queries = queries.reshape(-1, queries.shape[-1])
    Q = o_idx.shape[0]
    assert g_idx.shape == o_idx.shape, (g_idx.shape, o_idx.shape)
    swaps = 0
    for qi in range(Q):
        gi, oi = g_idx[qi].astype(np.int64), o_idx[qi].astype(np.int64)
        gs, os_ = g_score[qi].astype(np.float64), o_score[qi]
        assert len(set(gi.tolist())) == len(gi), f"query {qi}: duplicate rows in result {gi}"
        # rank-wise score parity
        tol = REL_TOL * np.abs(os_) + ABS_FLOOR
        bad = np.abs(gs - os_) > tol
        assert not bad.any(), f"query {qi} ({metric}): scores differ at ranks {np.where(bad)[0][:5]}: {gs[bad][:5]} vs {os_[bad][:5]}"
        # ordering as returned: descending similarity / ascending distance
        if metric == "euclidean":
            assert (np.diff(gs) >= -1e-7 * np.maximum(1.0, np.abs(gs[1:]))).all(), f"query {qi}: distances not ascending"
        else:
            assert (np.diff(gs) <= 1e-7 * np.maximum(1.0, np.abs(gs[1:]))).all(), f"query {qi}: scores not descending"
        if (gi == oi).all():
            continue
        # identical sets in a different order, or boundary swaps: verify with exact scores
        ex = exact_scores_for(rows, queries[qi], gi - row_base, metric)
        scale = max(1.0, float(np.abs(os_).max()))
        assert np.abs(ex - os_).max() <= swap_eps * scale, (
            f"query {qi} ({metric}): index mismatch beyond fp32 noise: got {gi}, want {oi}, "
            f"exact scores of got {ex}, oracle {os_}")
        swaps += int((gi != oi).sum())
    return swaps


def torch_fp64_topk(n, d, q, k, metric, slice_rows, rows_of_slice):
    """Exact fp64 brute force at full size ON THE GPU (torch, fp64 matmul over row slices) — an arithmetic completely
    independent of the kernels under test.  rows_of_slice(lo, cnt) -> float32 cuda tensor [cnt, d].  Returns (idx [Q, k]
    int64 cpu, score [Q, k] float64 cpu) under the (score desc, row asc) / (distance asc, row asc) order."""
    import torch
    q64 = torch.from_numpy(np.asarray(q, dtype=np.float64)).cuda()
    qn = q64.norm(dim=1)
    best_s = best_i = None
    for lo in range(0, n, slice_rows):
        cnt = min(slice_rows, n - lo)
        x = rows_of_slice(lo, cnt).double()
        s = x @ q64.T  # [cnt, Q]
        if metric == "cosine":
            den = x.norm(dim=1)[:, None] * qn[None, :]
            s = torch.where(den > 0, s / den, torch.zeros_like(s))
        elif metric == "euclidean":
            s = -((x * x).sum(1)[:, None] + (q64 * q64).sum(1)[None, :] - 2.0 * s)
        kk = min(k + 8, cnt)
        v, i = torch.topk(s, kk, dim=0)  # [kk, Q]
        i = i + lo
        if best_s is None:
            best_s, best_i = v, i
        else:
            best_s, best_i = torch.cat([best_s, v]), torch.cat([best_i, i])
            keep = torch.topk(best_s, min(k + 8, best_s.shape[0]), dim=0).indices
            best_s, best_i = torch.gather(best_s, 0, keep), torch.gather(best_i, 0, keep)
        del x, s
    # final order: score desc, row asc
    bs, bi = best_s.T.cpu().numpy(), best_i.T.cpu().numpy()
    out_i = np.empty((bs.shape[0], k), dtype=np.int64)
    out_s = np.empty((bs.shape[0], k), dtype=np.float64)
    for r in range(bs.shape[0]):
        order = np.lexsort((bi[r], -bs[r]))[:k]
        out_i[r], out_s[r] = bi[r][order], bs[r][order]
    if metric == "euclidean":
        out_s = np.sqrt(np.maximum(-out_s, 0.0))
    return out_i, out_s
