"""Host-side mirror of gpu.ClusterIndex (pkg/gpu/kmeans.go) over the device kernels — SURVEY.md §8(f)4.

Same method names, argument meaning and error identities as the Go type.  The two data-parallel steps of Lloyd's
algorithm run on the GPU against the HBM-resident corpus, nothing is copied back but the assignment vector:
  * assignment  = `nk_index_assign_nearest`: the fused scan with the roles swapped (centroids are the indexed corpus,
    the corpus rows are the queries, k = 1)                                   — kmeans.go:458-546
  * update      = `nk_index_cluster_means`: float64 per-cluster sums on device  — kmeans.go:585-618
  * cluster-restricted search = `nk_search_clusters`: routing, member gather and the exact scan of the probed clusters'
    rows in one device call for a whole batch (the clustering is installed lazily, `nk_index_set_clusters`)
                                                                              — kmeans.go:816-895
  * k-means++ seeding = `nk_index_kmeanspp`: D² weighting over every row, one streaming pass per centroid that skips
    rows the triangle inequality rules out                                    — kmeans.go:364-427
Centroid bookkeeping (K x dim, tiny) stays on the host in the reference's arithmetic (float32 differences, float64
squares: squaredEuclidean kmeans.go:430-454).

Deviations, stated: the reference seeds k-means++ / random init from Go's global math/rand stream, which cannot be
reproduced; this mirror takes a numpy Generator (seedable): k-means++ draws the first row and then one uniform variate
per centroid from it.  Only index stand-ins without `kmeanspp` seed on the host (`_init_kmeanspp`), and above
`init_sample` rows they do so on a uniform sample of the rows read back.  `assign` selects which of the reference's two assignment rules
is used: "euclidean" (assignToCentroids, the CPU definition) or "cosine" (assignToCentroidsGPU, what the reference runs
when its GPU manager is enabled).
"""
from __future__ import annotations

import math
import time
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence

import numpy as np

from .embedding_index import EmbeddingIndex, ErrInvalidDimensions, SearchResult
from .knn import NK_MAX_K


class ErrInvalidK(ValueError):  # kmeans.go ErrInvalidK
    def __init__(self):
        super().__init__("gpu: invalid K value")


class ErrTooFewEmbeddings(ValueError):  # kmeans.go ErrTooFewEmbeddings
    def __init__(self):
        super().__init__("gpu: too few embeddings for clustering")


@dataclass
class KMeansConfig:  # kmeans.go:57-93
    NumClusters: int = 0
    MaxIterations: int = 100
    Tolerance: float = 0.0001
    InitMethod: str = "kmeans++"
    AutoK: bool = True
    DriftThreshold: float = 0.1
    MinClusterSize: int = 10


@dataclass
class ClusterStats:  # kmeans.go:96-107
    EmbeddingCount: int = 0
    NumClusters: int = 0
    AvgClusterSize: float = 0.0
    MinClusterSize: int = 0
    MaxClusterSize: int = 0
    Iterations: int = 0
    LastClusterTime: float = 0.0
    Clustered: bool = False


def optimalK(n: int) -> int:
    """sqrt(n/2) clamped to [10, 1000] — kmeans.go:323-332."""
    k = int(math.sqrt(float(n) / 2))
    return max(10, min(1000, k))


def squaredEuclidean(a: np.ndarray, b: np.ndarray) -> np.ndarray:
    """kmeans.go:430-454 on the host for K x dim sized inputs: float32 differences, float64 squares."""
    d = (np.asarray(a, dtype=np.float32) - np.asarray(b, dtype=np.float32)).astype(np.float64)
    return (d * d).sum(axis=-1)


class ClusterIndex(EmbeddingIndex):
    def __init__(self, dimensions: int, kmeansConfig: Optional[KMeansConfig] = None, devices: Sequence[int] = (0,),
                 assign: str = "euclidean", rng: Optional[np.random.Generator] = None, init_sample: int = 200_000):
        super().__init__(dimensions, metric="cosine", devices=devices, dtype="f32")  # kmeans.go:200-229
        if assign not in ("euclidean", "cosine"):
            raise ValueError("assign must be 'euclidean' (kmeans.go:458) or 'cosine' (kmeans.go:491)")
        self.config = kmeansConfig or KMeansConfig()
        self.assign_metric = assign
        self.rng = rng or np.random.default_rng()
        self.init_sample = int(init_sample)
        self.centroids: Optional[np.ndarray] = None      # [K x dim] float32
        self.assignments: Optional[np.ndarray] = None    # [N] int32
        self.clusterMap: Dict[int, List[int]] = {}
        self.pendingUpdates: List[tuple] = []
        self.updatesSinceCluster = 0
        self.clustered = False
        self.lastClusterTime = 0.0
        self.lastClusterDuration = 0.0
        self.iterations = 0
        self.clusterIterations = 0
        self.centroidDrift = 0.0
        self._dev_stale = True  # the device's copy of (centroids, assignments) must be re-installed before a routed search

    # ---- initialisation (kmeans.go:335-427) ------------------------------------------------------------------------
    def _init_rows(self, n: int) -> np.ndarray:
        if n <= self.init_sample:
            return self._ix.read_rows(0, n)
        pick = np.sort(self.rng.choice(n, size=self.init_sample, replace=False))
        return np.stack([self._ix.read_rows(int(r), 1)[0] for r in pick])

    def _init_random(self, k: int, rows: np.ndarray) -> np.ndarray:
        return rows[self.rng.choice(rows.shape[0], size=k, replace=False)].astype(np.float32, copy=True)

    def _init_kmeanspp(self, k: int, rows: np.ndarray) -> np.ndarray:
        m = rows.shape[0]
        cen = np.empty((k, self.dimensions), dtype=np.float32)
        cen[0] = rows[int(self.rng.integers(m))]
        mind = squaredEuclidean(rows, cen[0])
        for c in range(1, k):
            total = float(mind.sum())
            target = float(self.rng.random()) * total
            cum = np.cumsum(mind)
            sel = int(np.searchsorted(cum, target, side="left"))  # first i with cumWeight >= target
            if sel >= m:
                sel = m - 1
            cen[c] = rows[sel]
            mind = np.minimum(mind, squaredEuclidean(rows, cen[c]))
        return cen

    # ---- Lloyd iterations on device (kmeans.go:232-320) ---------------------------------------------------------------
    def Cluster(self, initial_centroids=None) -> None:
        with self.mu:
            n = len(self.nodeIDs)
            if n == 0:
                return
            k = self.config.NumClusters
            if k <= 0 or self.config.AutoK:
                k = optimalK(n)
            if k > n:
                k = n
            if k < 1:
                raise ErrInvalidK()
            start = time.time()
            if initial_centroids is not None:
                cen = np.array(initial_centroids, dtype=np.float32, order="C", copy=True)
                if cen.shape != (k, self.dimensions):
                    raise ValueError(f"initial_centroids must be [{k} x {self.dimensions}]")
            elif self.config.InitMethod == "kmeans++" and hasattr(self._ix, "kmeanspp"):
                # every row takes part (kmeans.go:364-427); the same draws, in the same order, as _init_kmeanspp takes
                first = int(self.rng.integers(n))
                cen, _, _ = self._ix.kmeanspp(k, first, self.rng.random(k - 1))
            else:
                rows = self._init_rows(n)
                cen = self._init_kmeanspp(k, rows) if self.config.InitMethod == "kmeans++" else self._init_random(k, rows)
            assign = np.zeros(n, dtype=np.int32)  # make([]int, n)
            self.iterations = 0
            for _ in range(self.config.MaxIterations):
                changed = self._ix.assign_nearest(cen, assign, metric=self.assign_metric)
                cen, _ = self._ix.cluster_means(assign, cen)
                self.iterations += 1
                self.clusterIterations += 1
                if changed == 0:
                    break
            self.centroids, self.assignments = cen, assign
            self._dev_stale = True
            self._build_cluster_map()
            self.clustered = True
            self.lastClusterTime = time.time()
            self.lastClusterDuration = self.lastClusterTime - start
            self.updatesSinceCluster = 0

    def _build_cluster_map(self) -> None:  # kmeans.go:621-628 (members in ascending embedding index)
        self.clusterMap = {}
        order = np.argsort(self.assignments, kind="stable")
        bounds = np.searchsorted(self.assignments[order], np.arange(self.centroids.shape[0] + 1))
        for c in range(self.centroids.shape[0]):
            if bounds[c + 1] > bounds[c]:
                self.clusterMap[c] = order[bounds[c]:bounds[c + 1]].tolist()

    def Clear(self) -> None:  # kmeans.go:631-648
        with self.mu:
            super().Clear()
            self.centroids = None
            self.assignments = None
            self.clusterMap = {}
            self.pendingUpdates = []
            self.clustered = False
            self.updatesSinceCluster = 0
            self._dev_stale = True

    def IsClustered(self) -> bool:
        return self.clustered

    def NumClusters(self) -> int:
        return 0 if self.centroids is None else int(self.centroids.shape[0])

    def ClusterStats(self) -> ClusterStats:  # kmeans.go:665-701
        st = ClusterStats(EmbeddingCount=len(self.nodeIDs), NumClusters=self.NumClusters(), Iterations=self.iterations,
                          LastClusterTime=self.lastClusterTime, Clustered=self.clustered)
        if self.clustered and self.clusterMap:
            sizes = [len(m) for m in self.clusterMap.values()]
            st.AvgClusterSize = float(sum(sizes)) / len(sizes)
            st.MinClusterSize, st.MaxClusterSize = min(sizes), max(sizes)
        return st

    # ---- routing (kmeans.go:705-813) -----------------------------------------------------------------------------------
    def FindNearestCentroid(self, embedding) -> int:
        if not self.clustered or self.centroids is None or len(self.centroids) == 0:
            return -1
        return int(np.argmin(squaredEuclidean(self.centroids, np.asarray(embedding, dtype=np.float32))))  # first minimum

    def FindNearestClusters(self, embedding, k: int) -> Optional[List[int]]:
        if not self.clustered or self.centroids is None or len(self.centroids) == 0:
            return None
        k = min(int(k), len(self.centroids))
        d = squaredEuclidean(self.centroids, np.asarray(embedding, dtype=np.float32))
        return np.argsort(d, kind="stable")[:k].tolist()

    def GetClusterMembers(self, clusterIDs: Sequence[int]) -> Optional[List[int]]:
        if not self.clustered:
            return None
        members: List[int] = []
        for cid in clusterIDs:
            members.extend(self.clusterMap.get(int(cid), []))
        return members

    def SearchWithClusters(self, query, topK: int, numClusters: int) -> Optional[List[SearchResult]]:  # kmeans.go:816-836
        if not self.IsClustered():
            return self.Search(query, topK)
        q = np.asarray(query, dtype=np.float32).reshape(-1)
        if q.size != self.dimensions:
            raise ErrInvalidDimensions()
        return self.SearchWithClustersBatch(q.reshape(1, -1), topK, numClusters)[0]

    def SearchWithClustersBatch(self, queries, topK: int, numClusters: int) -> List[Optional[List[SearchResult]]]:
        """SearchWithClusters for every row of `queries` [Q x dim], one device call for the whole batch."""
        q = np.ascontiguousarray(np.asarray(queries, dtype=np.float32))
        if q.ndim != 2 or q.shape[1] != self.dimensions:
            raise ErrInvalidDimensions()
        if not self.IsClustered():
            return [self.Search(v, topK) for v in q]
        with self.mu:
            topK, numClusters = int(topK), int(numClusters)
            # the two cases the device call cannot serve: k above NK_MAX_K, and an assignment array that no longer covers
            # exactly the index's rows (Add without OnNodeUpdate, Remove: the reference leaves those inconsistent too).
            # KnnIndex always has search_clusters; an index stand-in that only scores subsets (the CPU test double of the
            # host-logic tests) is served by the same subset path the reference takes.
            if (numClusters <= 0 or topK <= 0 or topK > NK_MAX_K or len(self.assignments) != len(self._ix)
                    or not hasattr(self._ix, "search_clusters")):
                return [self._search_with_clusters_host(v, topK, numClusters) for v in q]
            if self._dev_stale:
                self._ix.set_clusters(self.centroids, self.assignments)
                self._dev_stale = False
            idx, sc = self._ix.search_clusters(q, topK, numClusters)
            out: List[Optional[List[SearchResult]]] = []
            for i in range(q.shape[0]):
                hit = idx[i] != 0xFFFFFFFF  # slots beyond the candidate count (topK clamped to it, kmeans.go:852-855)
                out.append([SearchResult(self.nodeIDs[int(r)], float(s), float(1.0 - s)) for r, s in zip(idx[i][hit], sc[i][hit])]
                           if hit.any() else None)
            return out

    def _search_with_clusters_host(self, q: np.ndarray, topK: int, numClusters: int) -> Optional[List[SearchResult]]:
        ids = self.FindNearestClusters(q, numClusters)
        if not ids:
            return None
        cand = self.GetClusterMembers(ids)
        if not cand:
            return None
        return self.SearchCandidates(q, cand, topK)

    # Row-count changing mutations clear the device's clustering: re-install it before the next routed search.
    def Add(self, nodeID: str, embedding) -> None:
        with self.mu:
            self._dev_stale = True
            super().Add(nodeID, embedding)

    def AddBatch(self, nodeIDs: Sequence[str], embeddings) -> None:
        with self.mu:
            self._dev_stale = True
            super().AddBatch(nodeIDs, embeddings)

    def Remove(self, nodeID: str) -> bool:
        with self.mu:
            self._dev_stale = True
            return super().Remove(nodeID)

    def Deserialize(self, data: bytes) -> None:
        with self.mu:
            self._dev_stale = True
            super().Deserialize(data)

    def SearchCandidates(self, query, candidateIndices: Sequence[int], topK: int) -> Optional[List[SearchResult]]:  # kmeans.go:839-895
        q = np.asarray(query, dtype=np.float32).reshape(-1)
        if q.size != self.dimensions:
            raise ErrInvalidDimensions()
        with self.mu:
            if len(candidateIndices) == 0:
                return None
            topK = min(int(topK), len(candidateIndices))
            if topK <= 0:
                return []
            idx, sc = self._ix.score_subset(q, list(candidateIndices), topK)
            return [SearchResult(self.nodeIDs[int(i)], float(s), float(1.0 - s)) for i, s in zip(idx, sc)]

    # ---- real-time updates (kmeans.go:910-1052) ---------------------------------------------------------------------
    def OnNodeUpdate(self, nodeID: str, embedding) -> None:
        self.Add(nodeID, embedding)
        if not self.IsClustered():
            return
        with self.mu:
            idx = self.idToIndex.get(nodeID)
            if idx is None:
                return
            new = self.FindNearestCentroid(embedding)
            if idx < len(self.assignments):
                old = int(self.assignments[idx])
                if new != old:
                    if old in self.clusterMap and idx in self.clusterMap[old]:
                        self.clusterMap[old].remove(idx)
                    self.clusterMap.setdefault(new, []).append(idx)
                    self.assignments[idx] = new
                    self.pendingUpdates.append((idx, old, new))
            else:
                self.assignments = np.append(self.assignments, np.int32(new))
                self.clusterMap.setdefault(new, []).append(idx)
            self.updatesSinceCluster += 1
            self._dev_stale = True

    def ShouldRecluster(self) -> bool:  # kmeans.go:980-1005
        if not self.clustered:
            return False
        if self.updatesSinceCluster / max(len(self.nodeIDs), 1) > 0.1:
            return True
        if self.centroidDrift > self.config.DriftThreshold:
            return True
        return time.time() - self.lastClusterTime > 3600.0

    def UpdateCentroidsBatch(self) -> None:  # kmeans.go:1009-1052: recompute the centroids of the affected clusters
        with self.mu:
            updates, self.pendingUpdates = self.pendingUpdates, []
            if not updates:
                return
            affected = {c for _, old, new in updates for c in (old, new)}
            fresh, counts = self._ix.cluster_means(self.assignments, self.centroids)
            for c in affected:
                if counts[c] > 0:
                    self.centroids[c] = fresh[c]
            self._dev_stale = True

    def Dimensions(self) -> int:
        return self.dimensions

    def GetConfig(self) -> KMeansConfig:
        return self.config
