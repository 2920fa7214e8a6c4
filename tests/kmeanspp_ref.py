"""References for nk_index_kmeanspp (k-means++ seeding, pkg/gpu/kmeans.go:364-427), test infrastructure only:

* `seq`: the sequential loop in C (kmeanspp_ref.c), compiled on first use into a temporary directory (the source tree may be
  read-only), loaded through ctypes;
* `transliteration`: the same loop in plain Python, line for line, for tiny inputs;
* `margins`: per step, how far the target lies from the nearest cumulative boundary (fp64, relative to the total), so a
  disagreement that comes from a rounding tie is told apart from a wrong selection.

The random numbers are injected: `first` stands for rand.Intn(n) and draws[c-1] for the c-th rand.Float64()."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def _load():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="kmeanspp_ref_"), "libkmeanspp_ref.so")
        subprocess.run(["/usr/bin/gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC", os.path.join(_HERE, "kmeanspp_ref.c"),
                        "-o", out], check=True)
        lib = C.CDLL(out)
        lib.ref_kmeanspp.restype = C.c_int
        lib.ref_kmeanspp.argtypes = [C.c_void_p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = lib
    return _lib


def seq(rows, K, first, draws):
    """(centroids float32 [K x dim], rows uint32 [K]) of the sequential loop."""
    r = np.ascontiguousarray(rows, dtype=np.float32)
    d = np.ascontiguousarray(np.asarray(draws, dtype=np.float64).reshape(-1))
    assert d.size == K - 1
    cen = np.empty((K, r.shape[1]), dtype=np.float32)
    out = np.empty(K, dtype=np.uint32)
    rc = _load().ref_kmeanspp(r.ctypes.data, r.shape[0], r.shape[1], K, int(first), d.ctypes.data if d.size else None,
                              cen.ctypes.data, out.ctypes.data)
    assert rc == 0
    return cen, out


def _sq_euclid(a, b):  # squaredEuclidean, kmeans.go:430-454
    n = len(a)
    s = [0.0, 0.0, 0.0, 0.0]
    i = 0
    while i <= n - 4:
        for j in range(4):
            d = float(np.float32(a[i + j]) - np.float32(b[i + j]))
            s[j] += d * d
        i += 4
    while i < n:
        d = float(np.float32(a[i]) - np.float32(b[i]))
        s[0] += d * d
        i += 1
    return s[0] + s[1] + s[2] + s[3]


def transliteration(rows, K, first, draws):
    """initCentroidsKMeansPlusPlus in plain Python: returns the selected rows (list of ints)."""
    with np.errstate(invalid="ignore", over="ignore"):  # NaN / Inf rows are part of the contract
        return _transliteration(np.asarray(rows, dtype=np.float32), K, first, draws)


def _transliteration(rows, K, first, draws):
    n = rows.shape[0]
    picked = [int(first)]
    min_d = [_sq_euclid(rows[i], rows[first]) for i in range(n)]
    for c in range(1, K):
        total = 0.0
        for i in range(n):
            total += min_d[i]
        target = float(draws[c - 1]) * total
        cum, sel = 0.0, n - 1
        for i in range(n):
            cum += min_d[i]
            if cum >= target:
                sel = i
                break
        picked.append(sel)
        for i in range(n):
            d = _sq_euclid(rows[i], rows[sel])
            if d < min_d[i]:
                min_d[i] = d
    return picked


def margins(rows, picked, draws):
    """For each step c >= 1 of a seeding that picked `picked`: min |cumsum_i - target| / total over the boundaries, from
    fp64 distances (float32 differences).  0 means the target sits exactly on a boundary; inf/NaN totals give NaN."""
    r = np.asarray(rows, dtype=np.float32)
    diff = r - r[picked[0]]
    mind = (diff.astype(np.float64) ** 2).sum(axis=1)
    out = []
    for c in range(1, len(picked)):
        with np.errstate(invalid="ignore", over="ignore"):
            total = mind.sum()
            cum = np.cumsum(mind)
            target = float(draws[c - 1]) * total
            out.append(float(np.min(np.abs(cum - target)) / total) if np.isfinite(total) and total > 0 else float("nan"))
        if c + 1 < len(picked):
            d = ((r - r[picked[c]]).astype(np.float64) ** 2).sum(axis=1)
            mind = np.where(d < mind, d, mind)
    return np.array(out)


def explain(got_rows, want_rows, rows, draws) -> str:
    """Message for a mismatch: the first step that differs and the margin of its target."""
    got_rows, want_rows = np.asarray(got_rows), np.asarray(want_rows)
    bad = np.flatnonzero(got_rows != want_rows)
    if bad.size == 0:
        return "identical"
    c = int(bad[0])
    m = margins(rows, [int(x) for x in want_rows[:c + 1]], draws) if c > 0 else np.array([])
    return (f"first difference at step {c}: device row {int(got_rows[c])}, reference row {int(want_rows[c])}; "
            f"target margin there {m[-1] if m.size else float('nan'):.3e} of the total")
