"""KnnIndex — thin host wrapper over the fused batched C ABI (nk_* in include/nornic_knn.h).

This is the object gpu.EmbeddingIndex would hold instead of a cuda.Buffer (pkg/gpu/gpu.go:1224-1260): a
row-major corpus resident in HBM, row-sharded across the GPUs of this process, searched Q queries at a
time by one fused distance + top-k kernel per shard."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np

from . import _lib

METRICS = {"cosine": 0, "dot": 1, "euclidean": 2}
DTYPES = {"f32": 0, "fp32": 0, "float32": 0, "f16": 1, "fp16": 1, "float16": 1, "bf16": 2, "bfloat16": 2}
PATHS = {"auto": 0, "simt": 1, "tensor": 2, "filter": 3, "shadow": 4}
NK_MAX_K = 1024
NK_MAX_CLUSTERS = 4096


class KnnError(RuntimeError):
    pass


def _check(ret: int, what: str) -> int:
    if ret < 0:
        raise KnnError(f"{what}: {_lib.last_error()}")
    return ret


class KnnIndex:
    def __init__(self, dim: int, metric: str = "cosine", dtype: str = "f32", devices: Sequence[int] = (0,)):
        self.lib = _lib.load()
        self.dim = int(dim)
        self.metric = metric
        self.dtype = DTYPES[dtype]
        # bf16 rows travel as raw uint16 bit patterns (numpy has no bfloat16): see to_bf16_bits / from_bf16_bits
        self.np_dtype = np.float16 if self.dtype == 1 else np.uint16 if self.dtype == 2 else np.float32
        self.devices = list(devices)
        self._clusters_k = 0  # K of the last clustering installed (nk_index_set_clusters)
        ids = (C.c_int * len(self.devices))(*self.devices)
        self.ptr = self.lib.nk_index_create(ids, len(self.devices), self.dim, self.dtype, METRICS[metric])
        if not self.ptr:
            raise KnnError(f"nk_index_create: {_lib.last_error()}")

    # -- lifecycle ---------------------------------------------------------------------------------
    def release(self) -> None:
        if self.ptr:
            self.lib.nk_index_release(self.ptr)
            self.ptr = None

    close = release

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def __len__(self) -> int:
        return int(self.lib.nk_index_rows(self.ptr))

    # -- corpus ------------------------------------------------------------------------------------
    def _rows(self, rows) -> np.ndarray:
        if self.dtype == 2 and np.asarray(rows).dtype.kind == "f":
            rows = to_bf16_bits(rows)  # float input to a bf16 index: round to nearest even, like the device does
        a = np.ascontiguousarray(np.asarray(rows, dtype=self.np_dtype))
        if a.size % self.dim:
            raise KnnError("rows are not a multiple of dim")
        return a.reshape(-1, self.dim)

    def upload(self, rows) -> None:
        a = self._rows(rows)
        _check(self.lib.nk_index_upload(self.ptr, a.ctypes.data_as(C.c_void_p), a.shape[0]), "nk_index_upload")

    def upload_from_f32(self, rows=None, ptr: Optional[int] = None, n_rows: Optional[int] = None) -> None:
        """Upload fp32 host rows whatever the dtype of the index (fp16 indexes convert on the device while loading).
        Either a [n x dim] array, or a raw host address + row count (e.g. the payload of a serialized index)."""
        if ptr is None:
            a = np.ascontiguousarray(np.asarray(rows, dtype=np.float32)).reshape(-1, self.dim)
            ptr, n_rows = a.ctypes.data, a.shape[0]
        _check(self.lib.nk_index_upload_from_f32(self.ptr, C.c_void_p(ptr), int(n_rows)), "nk_index_upload_from_f32")

    def set_row_mask(self, keep) -> None:
        """Row filter for the following searches: `keep` = boolean array with one entry per row (True = may be returned),
        or None to clear.  (Label filter of queryNodes, call_vector.go:177-193, evaluated inside the scan kernels.)"""
        if keep is None:
            _check(self.lib.nk_index_set_row_mask(self.ptr, None, 0), "nk_index_set_row_mask")
            return
        b = np.asarray(keep, dtype=bool).reshape(-1)
        words = np.packbits(b, bitorder="little")
        words = np.concatenate([words, np.zeros((-len(words)) % 4, dtype=np.uint8)]).view("<u4")
        words = np.ascontiguousarray(words)
        _check(self.lib.nk_index_set_row_mask(self.ptr, words.ctypes.data_as(C.c_void_p), int(b.size)), "nk_index_set_row_mask")

    def append(self, rows) -> None:
        a = self._rows(rows)
        _check(self.lib.nk_index_append(self.ptr, a.ctypes.data_as(C.c_void_p), a.shape[0]), "nk_index_append")

    def update_row(self, row: int, vec) -> None:
        a = self._rows(vec)
        _check(self.lib.nk_index_update_row(self.ptr, int(row), a.ctypes.data_as(C.c_void_p)), "nk_index_update_row")

    def remove_swap(self, row: int) -> None:
        _check(self.lib.nk_index_remove_swap(self.ptr, int(row)), "nk_index_remove_swap")

    def fill_uniform(self, n_rows: int, seed: int) -> None:
        _check(self.lib.nk_index_fill_uniform(self.ptr, int(n_rows), int(seed)), "nk_index_fill_uniform")

    def fill_clustered(self, n_rows: int, seed: int, n_centres: int = 1000, sigma: float = 0.1, unit_norm: bool = False) -> None:
        """SURVEY.md 8(d)'s Gaussian-mixture corpus, generated on the device (near-tie stress case)."""
        _check(self.lib.nk_index_fill_clustered(self.ptr, int(n_rows), int(seed), int(n_centres), float(sigma), 1 if unit_norm else 0),
               "nk_index_fill_clustered")

    def refresh_shadow(self) -> None:
        _check(self.lib.nk_index_refresh_shadow(self.ptr), "nk_index_refresh_shadow")

    def set_metric(self, metric: str) -> None:
        _check(self.lib.nk_index_set_metric(self.ptr, METRICS[metric]), "nk_index_set_metric")
        self.metric = metric

    def set_min_score(self, min_score: Optional[float]) -> None:
        """Score floor evaluated inside the kernels (cosine / dot: minimum similarity; euclidean: maximum distance).
        None clears it."""
        if min_score is None:
            min_score = float("inf") if self.metric == "euclidean" else float("-inf")
        _check(self.lib.nk_index_set_min_score(self.ptr, float(min_score)), "nk_index_set_min_score")

    def set_row_groups(self, group_of_row, n_groups: Optional[int] = None) -> None:
        if group_of_row is None:
            _check(self.lib.nk_index_set_row_groups(self.ptr, None, 0, 0), "nk_index_set_row_groups")
            return
        g = np.ascontiguousarray(np.asarray(group_of_row, dtype=np.uint32).reshape(-1))
        ng = int(g.max()) + 1 if n_groups is None and g.size else int(n_groups or 1)
        _check(self.lib.nk_index_set_row_groups(self.ptr, g.ctypes.data_as(C.c_void_p), int(g.size), ng), "nk_index_set_row_groups")

    def search_groups(self, query, k: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Best-of-chunks per node: (node ids, rows of their best chunks, scores), best first."""
        q = np.ascontiguousarray(np.asarray(query, dtype=np.float32).reshape(-1))
        if q.size != self.dim:
            raise KnnError(f"invalid dimensions: query has {q.size}, index has {self.dim}")
        k = int(k)
        if k <= 0:
            return np.empty(0, np.uint32), np.empty(0, np.uint32), np.empty(0, np.float32)
        grp = np.empty(k, dtype=np.uint32); row = np.empty(k, dtype=np.uint32); sc = np.empty(k, dtype=np.float32)
        n = _check(self.lib.nk_search_groups(self.ptr, q.ctypes.data_as(C.c_void_p), k, grp.ctypes.data_as(C.c_void_p),
                                             row.ctypes.data_as(C.c_void_p), sc.ctypes.data_as(C.c_void_p)), "nk_search_groups")
        return grp[:n], row[:n], sc[:n]

    def debug_counters(self) -> dict:
        out = (C.c_uint64 * 4)()
        _check(self.lib.nk_index_debug_counters(self.ptr, out), "nk_index_debug_counters")
        return {"bf16_stage_retries": int(out[0]), "exact_stage_runs": int(out[1]), "longest_list": int(out[2]), "overflow_bits": int(out[3])}

    def filter_dump(self, queries, which: str = "shadow") -> Tuple[np.ndarray, np.ndarray]:
        """Tests only: (estimate, bound) arrays [rows x Q] of the filter kernel `which` ("shadow" | "filter")."""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32)).reshape(-1, self.dim)
        n = len(self)
        est = np.empty((n, q.shape[0]), dtype=np.float32)
        bnd = np.empty((n, q.shape[0]), dtype=np.float32)
        _check(self.lib.nk_debug_filter_dump(self.ptr, q.ctypes.data_as(C.c_void_p), q.shape[0], PATHS[which],
                                             est.ctypes.data_as(C.c_void_p), bnd.ctypes.data_as(C.c_void_p)), "nk_debug_filter_dump")
        return est, bnd

    def status(self, stream: int = 0) -> None:
        _check(self.lib.nk_index_status(self.ptr, stream), "nk_index_status")

    def search_sharded_device(self, comm: "Comm", q_ptr: int, Q: int, k: int, out_idx_ptr: int, out_score_ptr: int, stream: int = 0) -> int:
        return _check(self.lib.nk_search_sharded_device(self.ptr, comm.ptr, q_ptr, Q, k, out_idx_ptr, out_score_ptr, stream),
                      "nk_search_sharded_device")

    def set_row_base(self, row_base: int) -> None:
        _check(self.lib.nk_index_set_row_base(self.ptr, int(row_base)), "nk_index_set_row_base")

    def attach_device_rows(self, dev_ptr: int, n_rows: int) -> None:
        _check(self.lib.nk_index_attach_device_rows(self.ptr, int(dev_ptr), int(n_rows)), "nk_index_attach_device_rows")

    def set_path(self, path: str) -> None:
        _check(self.lib.nk_index_set_path(self.ptr, PATHS[path]), "nk_index_set_path")

    def read_rows(self, row: int, n_rows: int) -> np.ndarray:
        out = np.empty((n_rows, self.dim), dtype=self.np_dtype)
        _check(self.lib.nk_index_read_rows(self.ptr, int(row), int(n_rows), out.ctypes.data_as(C.c_void_p)),
               "nk_index_read_rows")
        return out

    def debug_flags(self):
        out = (C.c_int * 4)()
        _check(self.lib.nk_index_debug_flags(self.ptr, out), "nk_index_debug_flags")
        return [int(v) for v in out]

    def last_path(self) -> str:
        return {1: "simt", 2: "tensor", 3: "filter", 4: "shadow"}.get(int(self.lib.nk_index_last_path(self.ptr)), "?")

    def enable_timing(self, on: bool = True) -> None:
        _check(self.lib.nk_index_enable_timing(self.ptr, 1 if on else 0), "nk_index_enable_timing")

    def scan_time_ms(self) -> Tuple[float, int]:
        ms, n = C.c_double(0), C.c_uint64(0)
        _check(self.lib.nk_index_scan_time_ms(self.ptr, C.byref(ms), C.byref(n)), "nk_index_scan_time_ms")
        return float(ms.value), int(n.value)

    def stats(self) -> dict:
        st = _lib.NkStats()
        _check(self.lib.nk_index_stats(self.ptr, C.byref(st)), "nk_index_stats")
        return {name: int(getattr(st, name)) for name, _ in st._fields_}

    # -- search ------------------------------------------------------------------------------------
    def search(self, queries, k: int) -> Tuple[np.ndarray, np.ndarray]:
        """queries [Q x dim] fp32 host -> (idx [Q x k'] uint32, score [Q x k'] fp32), k' = min(k, N).
        Euclidean scores are distances (ascending); cosine / dot are similarities (descending)."""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32))
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.shape[1] != self.dim:
            raise KnnError(f"invalid dimensions: query has {q.shape[1]}, index has {self.dim}")  # gpu.go:1533-1535
        Q = q.shape[0]
        k = int(k)
        if k <= 0 or Q == 0:
            return np.empty((Q, 0), np.uint32), np.empty((Q, 0), np.float32)
        idx = np.empty((Q, k), dtype=np.uint32)
        sc = np.empty((Q, k), dtype=np.float32)
        ke = _check(self.lib.nk_search(self.ptr, q.ctypes.data_as(C.c_void_p), Q, k, idx.ctypes.data_as(C.c_void_p),
                                       sc.ctypes.data_as(C.c_void_p)), "nk_search")
        return idx[:, :ke], sc[:, :ke]

    def search_device(self, q_ptr: int, Q: int, k: int, out_idx_ptr: int, out_score_ptr: int, stream: int = 0) -> int:
        return _check(self.lib.nk_search_device(self.ptr, q_ptr, Q, k, out_idx_ptr, out_score_ptr, stream),
                      "nk_search_device")

    def search_keys_device(self, q_ptr: int, Q: int, k: int, out_keys_ptr: int, stream: int = 0) -> int:
        return _check(self.lib.nk_search_keys_device(self.ptr, q_ptr, Q, k, out_keys_ptr, stream),
                      "nk_search_keys_device")

    def score_subset(self, query, rows: Sequence[int], k: Optional[int] = None) -> Tuple[np.ndarray, np.ndarray]:
        q = np.ascontiguousarray(np.asarray(query, dtype=np.float32).reshape(-1))
        if q.size != self.dim:
            raise KnnError(f"invalid dimensions: query has {q.size}, index has {self.dim}")
        r = np.ascontiguousarray(np.asarray(rows, dtype=np.uint32).reshape(-1))
        kk = len(r) if k is None else min(int(k), len(r))
        if kk <= 0:
            return np.empty(0, np.uint32), np.empty(0, np.float32)
        idx = np.empty(kk, dtype=np.uint32)
        sc = np.empty(kk, dtype=np.float32)
        ke = _check(self.lib.nk_score_subset(self.ptr, q.ctypes.data_as(C.c_void_p), r.ctypes.data_as(C.c_void_p),
                                             len(r), kk, idx.ctypes.data_as(C.c_void_p),
                                             sc.ctypes.data_as(C.c_void_p)), "nk_score_subset")
        return idx[:ke], sc[:ke]

    # ---- cluster-routed search (ClusterIndex.SearchWithClusters, kmeans.go:816-836) -------------------------------
    def set_clusters(self, centroids, assign) -> None:
        """Install a clustering for search_clusters: centroids [K x dim] and one int32 assignment per row (values outside
        [0, K) belong to no cluster).  None clears.  Row-count changing mutations clear it; update_row keeps it."""
        if centroids is None:
            _check(self.lib.nk_index_set_clusters(self.ptr, None, 0, None, 0), "nk_index_set_clusters")
            self._clusters_k = 0
            return
        c = np.ascontiguousarray(np.asarray(centroids, dtype=np.float32))
        if c.ndim != 2 or c.shape[1] != self.dim:
            raise KnnError(f"invalid dimensions: centroids {c.shape}, index has {self.dim}")
        a = np.ascontiguousarray(np.asarray(assign, dtype=np.int32).reshape(-1))
        _check(self.lib.nk_index_set_clusters(self.ptr, c.ctypes.data_as(C.c_void_p), c.shape[0], a.ctypes.data_as(C.c_void_p), a.size),
               "nk_index_set_clusters")
        self._clusters_k = c.shape[0]

    def search_clusters(self, queries, k: int, n_probe: int, return_probes: bool = False):
        """Route each query to its n_probe nearest centroids and search their members exactly.  Returns (idx [Q x k'],
        score [Q x k']) with k' = min(k, rows), and the probe lists [Q x min(n_probe, K)] when return_probes."""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32))
        if q.ndim == 1:
            q = q.reshape(1, -1)
        if q.shape[1] != self.dim:
            raise KnnError(f"invalid dimensions: query has {q.shape[1]}, index has {self.dim}")
        Q, k, n_probe = q.shape[0], int(k), int(n_probe)
        idx = np.empty((Q, max(k, 0)), dtype=np.uint32)
        sc = np.empty((Q, max(k, 0)), dtype=np.float32)
        probes = np.empty((Q, max(n_probe, 0)), dtype=np.int32)
        ke = _check(self.lib.nk_search_clusters(self.ptr, q.ctypes.data_as(C.c_void_p), Q, max(k, 0), max(n_probe, 0),
                                                idx.ctypes.data_as(C.c_void_p), sc.ctypes.data_as(C.c_void_p),
                                                probes.ctypes.data_as(C.c_void_p)), "nk_search_clusters")
        if not return_probes:
            return idx[:, :ke], sc[:, :ke]
        P = min(n_probe, self._clusters_k) if ke else 0  # the probe lists are packed with row stride P
        return idx[:, :ke], sc[:, :ke], probes.reshape(-1)[:Q * P].reshape(Q, P)

    def search_clusters_device(self, q_ptr: int, Q: int, k: int, n_probe: int, out_idx_ptr: int, out_score_ptr: int,
                               out_probe_ptr: int = 0, stream: int = 0) -> int:
        """Device-resident, asynchronous on `stream`: out arrays [Q x k] (and [Q x min(n_probe, K)] probes, optional)."""
        return _check(self.lib.nk_search_clusters_device(self.ptr, q_ptr, Q, k, n_probe, out_idx_ptr, out_score_ptr, out_probe_ptr or None,
                                                         stream), "nk_search_clusters_device")

    # ---- k-means routing on device (pkg/gpu/kmeans.go) ----------------------------------------------------------
    def assign_nearest(self, centroids, assign: np.ndarray, metric: str = "euclidean") -> int:
        """assignToCentroids (euclidean) / assignToCentroidsGPU (cosine): `assign` (int32 [rows]) is updated in place,
        returns the number of changed assignments."""
        c = np.ascontiguousarray(np.asarray(centroids, dtype=np.float32))
        if c.ndim != 2 or c.shape[1] != self.dim:
            raise KnnError(f"invalid dimensions: centroids {c.shape}, index has {self.dim}")
        if assign.dtype != np.int32 or not assign.flags.c_contiguous or assign.size != len(self):
            raise KnnError("assign must be a contiguous int32 array with one entry per row")
        changed = C.c_uint64(0)
        _check(self.lib.nk_index_assign_nearest(self.ptr, c.ctypes.data_as(C.c_void_p), c.shape[0], METRICS[metric],
                                                assign.ctypes.data_as(C.c_void_p), C.byref(changed)), "nk_index_assign_nearest")
        return int(changed.value)

    def cluster_means(self, assign: np.ndarray, centroids) -> Tuple[np.ndarray, np.ndarray]:
        """updateCentroidsWithBuffer: returns (new centroids float32 [K x dim], member counts uint32 [K])."""
        c = np.array(centroids, dtype=np.float32, order="C", copy=True)
        a = np.ascontiguousarray(assign, dtype=np.int32)
        if a.size != len(self):
            raise KnnError("assign must have one entry per row")
        counts = np.zeros(c.shape[0], dtype=np.uint32)
        _check(self.lib.nk_index_cluster_means(self.ptr, a.ctypes.data_as(C.c_void_p), c.shape[0], c.ctypes.data_as(C.c_void_p),
                                               counts.ctypes.data_as(C.c_void_p)), "nk_index_cluster_means")
        return c, counts

    def kmeanspp(self, K: int, first_row: int, draws) -> Tuple[np.ndarray, np.ndarray, int]:
        """initCentroidsKMeansPlusPlus over every row, on the device: centroid 0 is row `first_row`, centroid c is chosen
        by the uniform variate draws[c-1] in [0, 1).  Returns (centroids float32 [K x dim], their rows uint32 [K], how
        many (row, step) distances were computed rather than skipped)."""
        K = int(K)
        d = np.ascontiguousarray(np.asarray(draws, dtype=np.float64).reshape(-1))
        if K >= 1 and d.size != K - 1:
            raise KnnError(f"kmeanspp: {d.size} draws for K={K} (need K - 1)")
        cen = np.empty((max(K, 0), self.dim), dtype=np.float32)
        rows = np.empty(max(K, 0), dtype=np.uint32)
        scored = C.c_uint64(0)
        _check(self.lib.nk_index_kmeanspp(self.ptr, max(K, 0), int(first_row), d.ctypes.data_as(C.c_void_p) if d.size else None,
                                          cen.ctypes.data_as(C.c_void_p), rows.ctypes.data_as(C.c_void_p), C.byref(scored)),
               "nk_index_kmeanspp")
        return cen, rows, int(scored.value)


def to_bf16_bits(a) -> np.ndarray:
    """fp32 array -> bf16 bit patterns (uint16), round to nearest even (what the device conversion does)."""
    u = np.ascontiguousarray(np.asarray(a, dtype=np.float32)).view(np.uint32)
    r = ((u >> 16) & 1) + np.uint32(0x7FFF)
    return ((u + r) >> 16).astype(np.uint16)


def from_bf16_bits(b) -> np.ndarray:
    return (np.asarray(b, dtype=np.uint16).astype(np.uint32) << 16).view(np.float32)


class Comm:
    """One rank's exchange context of a row-sharded search (nk_comm_*): candidate lists cross GPUs by peer stores."""

    def __init__(self, device: int, rank: int, world: int, slot_bytes: int):
        self.lib = _lib.load()
        self.rank, self.world = rank, world
        self.ptr = self.lib.nk_comm_create(int(device), int(rank), int(world), int(slot_bytes))
        if not self.ptr:
            raise KnnError(f"nk_comm_create: {_lib.last_error()}")

    def export(self) -> bytes:
        buf = C.create_string_buffer(64)
        _check(self.lib.nk_comm_export(self.ptr, buf), "nk_comm_export")
        return bytes(buf.raw)

    def connect(self, handles: Sequence[bytes]) -> None:
        blob = b"".join(handles)
        assert len(blob) == 64 * self.world
        _check(self.lib.nk_comm_connect(self.ptr, C.c_char_p(blob)), "nk_comm_connect")

    @staticmethod
    def connect_local(comms: Sequence["Comm"]) -> None:
        arr = (C.c_void_p * len(comms))(*[c.ptr for c in comms])
        _check(_lib.load().nk_comm_connect_local(arr, len(comms)), "nk_comm_connect_local")

    def status(self, stream: int = 0) -> None:
        _check(self.lib.nk_comm_status(self.ptr, stream), "nk_comm_status")

    def release(self) -> None:
        if self.ptr:
            self.lib.nk_comm_release(self.ptr)
            self.ptr = None


def blob_vectors(data: bytes) -> Tuple[int, int, int]:
    """(dims, count, byte offset of the fp32 vectors) of a serialized index (gpu.go:2373-2412)."""
    dims, count, off = C.c_uint32(0), C.c_uint32(0), C.c_size_t(0)
    _check(_lib.load().nk_blob_vectors(C.c_char_p(data), len(data), C.byref(dims), C.byref(count), C.byref(off)), "nk_blob_vectors")
    return int(dims.value), int(count.value), int(off.value)


def merge_keys_device(device_id: int, keys_ptr: int, n_lists: int, Q: int, k: int, metric: str, out_idx_ptr: int,
                      out_score_ptr: int, stream: int = 0) -> None:
    _check(_lib.load().nk_merge_keys_device(device_id, keys_ptr, n_lists, Q, k, METRICS[metric], out_idx_ptr,
                                            out_score_ptr, stream), "nk_merge_keys_device")


def fill_uniform_device(device_id: int, out_ptr: int, n_rows: int, dim: int, seed: int, row_base: int = 0,
                        stream: int = 0) -> None:
    _check(_lib.load().nk_fill_uniform_device(device_id, out_ptr, n_rows, dim, seed, row_base, stream),
           "nk_fill_uniform_device")
