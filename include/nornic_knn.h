/*
 * nornic_knn.h — C ABI of libnornic_knn.so, the B200-native brute-force kNN engine that sits behind
 * NornicDB's GPU boundary.
 *
 * Part 1 re-exports, symbol for symbol, the C functions of the cgo preamble in the reference's
 * pkg/gpu/cuda/cuda_bridge.go (lines cited per function) so that file can link this library instead
 * of carrying its own cuBLAS code (INTEGRATION.md shows the two-line change).  Part 2 is the fused,
 * batched API the Go host calls after a one-function change in cuda.Device.Search.
 *
 * Conventions (same as the reference, cuda_bridge.go:20-33,452-453): int returns are 0 = ok, -1 =
 * failure with a message retrievable through cuda_get_last_error() / nk_last_error(); pointer
 * returns are NULL on failure.  Unlike the reference's process-global buffer, the message is
 * thread-local.  Every entry point binds its CUDA device itself (cudaSetDevice per call), so
 * callers may migrate between OS threads (goroutines) freely.  Host pointers are only borrowed for
 * the duration of a call; every host-pointer entry point is synchronous.
 *
 * No torch / C++ types cross this boundary: plain pointers and sizes only.
 */
#ifndef NORNIC_KNN_H
#define NORNIC_KNN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ======================================================================================
 * Part 1 — legacy ABI (drop-in for the cgo preamble of pkg/gpu/cuda/cuda_bridge.go)
 * ====================================================================================== */

/* cuda_bridge.go:36-40.  Opaque to Go (only ever held as *C.CudaDevice).  The reference's struct
 * carries a cuBLAS handle; this library has no cuBLAS dependency. */
typedef struct CudaDevice CudaDevice;

/* cuda_bridge.go:132-136.  Field layout kept identical (data, size in BYTES, memory_type). */
typedef struct CudaBuffer {
    float *data;
    size_t size;
    int memory_type; /* 0 = device, 1 = pinned host */
} CudaBuffer;

void cuda_set_error(const char *msg);  /* cuda_bridge.go:23 */
const char *cuda_get_last_error(void); /* cuda_bridge.go:27 */
void cuda_clear_error(void);           /* cuda_bridge.go:31 */

int cuda_get_device_count(void);                     /* cuda_bridge.go:42  (-1 on error) */
int cuda_is_available(void);                         /* cuda_bridge.go:52  (1/0) */
CudaDevice *cuda_create_device(int device_id);       /* cuda_bridge.go:56  (NULL on error) */
void cuda_release_device(CudaDevice *dev);           /* cuda_bridge.go:94  (NULL-safe) */
const char *cuda_device_name(int device_id);         /* cuda_bridge.go:102 ("Unknown" on error) */
size_t cuda_device_memory(int device_id);            /* cuda_bridge.go:113 (bytes, 0 on error) */
int cuda_device_compute_capability(int device_id);   /* cuda_bridge.go:122 (major*10+minor; B200 = 100) */

/* cuda_bridge.go:138.  count is in floats; host_data may be NULL (uninitialised buffer); the copy
 * is synchronous.  memory_type 0 = device, 1 = pinned host. */
CudaBuffer *cuda_create_buffer(CudaDevice *dev, float *host_data, size_t count, int memory_type);
void cuda_release_buffer(CudaBuffer *buf);           /* cuda_bridge.go:184 (NULL-safe) */
void *cuda_buffer_data(CudaBuffer *buf);             /* cuda_bridge.go:197 */
size_t cuda_buffer_size(CudaBuffer *buf);            /* cuda_bridge.go:201 */
/* cuda_bridge.go:205.  Copies min(count*4, size) bytes; 0 / -1. */
int cuda_buffer_copy_to_host(CudaBuffer *buf, float *host_data, size_t count);

/* cuda_bridge.go:231.  norms[i] = ||vectors[i]||2.  One kernel (the reference issues n cublasSnrm2 calls). */
int cuda_compute_norms(CudaDevice *dev, CudaBuffer *vectors, CudaBuffer *norms, unsigned int n, unsigned int dims);
/* cuda_bridge.go:249.  In place; rows with norm <= 1e-10 are left untouched (cuda_bridge.go:267). */
int cuda_normalize_vectors(CudaDevice *dev, CudaBuffer *vectors, unsigned int n, unsigned int dims);
/* cuda_bridge.go:290.  scores[i] = embeddings[i] . query when normalized != 0 (what the reference's
 * sgemv computes for every input, cuda_bridge.go:293-309); when normalized == 0 the true cosine
 * dot/(|e||q|) with 0 for zero vectors (the case the reference leaves as a TODO). */
int cuda_cosine_similarity(CudaDevice *dev, CudaBuffer *embeddings, CudaBuffer *query, CudaBuffer *scores,
                           unsigned int n, unsigned int dims, int normalized);
/* cuda_bridge.go:327.  out_indices/out_scores are HOST arrays of length k; k is clamped to n; result
 * sorted by score descending, ties by lowest index first (the strict '>' forward scan of
 * cuda_bridge.go:356-371).  Selection runs on the device; only k pairs cross PCIe. */
int cuda_topk(CudaDevice *dev, CudaBuffer *scores, unsigned int *out_indices, float *out_scores, unsigned int n,
              unsigned int k);

/* ======================================================================================
 * Part 2 — fused batched kNN API (what cuda.Device.Search / gpu.EmbeddingIndex call instead of
 * NewBuffer + CosineSimilarity + TopK; SURVEY.md §8b)
 * ====================================================================================== */

/* Metric enum = vectorspace.DistanceMetric, pkg/vectorspace/registry.go:27-31. */
enum { NK_METRIC_COSINE = 0, NK_METRIC_DOT = 1, NK_METRIC_EUCLIDEAN = 2 };
/* Corpus element type held in HBM.  Queries and scores are always fp32.  fp16 / bf16 corpora (SURVEY.md §8(f)3 "fp16/bf16
 * down-conversion at load") are half the bytes; batches of >= 5 queries scan them IN PLACE on the tensor cores
 * (tcgen05.mma.kind::f16 with fp16 or bf16 operands — no shadow copy, no row-side rounding residue). */
enum { NK_DTYPE_F32 = 0, NK_DTYPE_F16 = 1, NK_DTYPE_BF16 = 2 };
/* Kernel selection for nk_index_set_path (diagnostics / tests); AUTO picks by Q, dim and dtype. */
/* TENSOR = exact 3xTF32 tensor-core scan; TENSOR_FILTER = 1xTF32 prefilter over the fp32 rows with rigorous margins +
 * exact fp32 rescoring (device-side fallback to the exact scan on margin overflow); TENSOR_SHADOW = the same filter
 * streaming a BF16 shadow copy of the shard (half the HBM bytes; built at upload for library-owned fp32 shards unless
 * NK_SHADOW=0, +50% device memory), exact fp32 rescoring from the fp32 rows, device-side retry through TENSOR_FILTER
 * and then the exact scan.  All paths return identical index sets. */
enum { NK_PATH_AUTO = 0, NK_PATH_SIMT = 1, NK_PATH_TENSOR = 2, NK_PATH_TENSOR_FILTER = 3, NK_PATH_TENSOR_SHADOW = 4 };

/* k up to NK_MAX_K is one fused pass; larger k (the reference accepts any k) is served by ceil(k/NK_MAX_K) passes
 * of the CUDA-core scan, up to NK_MAX_K_TOTAL results per query. */
#define NK_MAX_K 1024u
#define NK_MAX_K_TOTAL 65536u

typedef struct NkIndex NkIndex;
/* Exchange context of one rank of a row-sharded, one-rank-per-GPU search (see "Row-sharded search" below). */
typedef struct NkComm NkComm;
#define NK_COMM_HANDLE_BYTES 64 /* sizeof(cudaIpcMemHandle_t) */

typedef struct NkStats {
    uint64_t rows;            /* total rows resident */
    uint64_t searches;        /* nk_search* calls */
    uint64_t queries;         /* queries answered */
    uint64_t kernel_launches; /* kernels launched by this index */
    uint64_t bytes_h2d;       /* host->device bytes moved by this index */
    uint64_t bytes_d2h;
    uint64_t bytes_scanned;   /* corpus bytes streamed from HBM by search kernels */
    uint32_t n_devices;
    uint32_t dim;
} NkStats;

const char *nk_last_error(void);
const char *nk_version(void);

/* An index = one row-major [N x dim] corpus, row-sharded by contiguous ranges over n_devices GPUs of
 * this process (shard g holds rows [base_g, base_g + n_g)).  gpu.EmbeddingIndex storage, gpu.go:1224-1260. */
NkIndex *nk_index_create(const int *device_ids, int n_devices, uint32_t dim, int dtype, int metric);
void nk_index_release(NkIndex *ix); /* NULL-safe */

/* Replace the corpus with n_rows host rows (dtype of the index), split evenly over the devices.
 * Replaces syncToCUDA's NewBuffer + NormalizeVectors (gpu.go:2073-2118): rows are stored RAW; cosine
 * normalisation happens inside the search kernel, so device rows always equal host rows. */
int nk_index_upload(NkIndex *ix, const void *rows_host, uint64_t n_rows);
/* The same from fp32 host rows whatever the dtype of the index: an fp16 index converts on the device while loading
 * (round to nearest even).  Uploads stream through two pinned staging buffers, so pageable or unaligned sources load
 * at the PCIe / host-memcpy rate. */
int nk_index_upload_from_f32(NkIndex *ix, const float *rows_host_f32, uint64_t n_rows);
/* Locate the vectors inside a serialized index (EmbeddingIndex.Serialize, gpu.go:2373-2412: LE [dims u32][count u32]
 * [count x (len u32, id bytes)][count x dims fp32]) so that they can be fed straight to nk_index_upload_from_f32 —
 * the ids are the host language's business.  vec_offset has no alignment guarantee.  0 / -1 ("gpu: invalid
 * serialized data" for blobs shorter than the header, gpu.go:2419-2421). */
int nk_blob_vectors(const void *blob, size_t blob_bytes, uint32_t *dims, uint32_t *count, size_t *vec_offset);
/* Append rows to the last shard without re-uploading the rest (EmbeddingIndex.Add, gpu.go:1378-1434). */
int nk_index_append(NkIndex *ix, const void *rows_host, uint64_t n_rows);
/* Overwrite row `row` (global index) in place (EmbeddingIndex.Add on an existing id, gpu.go:1391-1399). */
int nk_index_update_row(NkIndex *ix, uint64_t row, const void *row_host);
/* Swap-with-last removal (EmbeddingIndex.Remove, gpu.go:1437-1471): row `row` takes the contents of the
 * last row and the corpus shrinks by one. */
int nk_index_remove_swap(NkIndex *ix, uint64_t row);
/* Row filter for subsequent searches — the label / type filter of db.index.vector.queryNodes (call_vector.go:177-193) as
 * a row bitmask, also usable for tombstones: bit r of mask_words (LSB first in 32-bit words, n_bits = rows of the index)
 * set = row r may be returned; k is clamped to the number of set bits.  NULL clears the filter.  Honoured inside every
 * scan kernel (no over-fetch).  upload / append / remove_swap / fill / attach clear it. */
int nk_index_set_row_mask(NkIndex *ix, const uint32_t *mask_words, uint64_t n_bits);
/* Fill the index with n_rows synthetic rows generated ON DEVICE by the counter-based generator shared
 * with the oracle (oracle/knn_oracle.c orc_fill_uniform): U[-1,1), element (r,j) depends only on
 * (seed, r, j).  Used by bench.py and the large-shape tests so 40 GB corpora never cross PCIe. */
int nk_index_fill_uniform(NkIndex *ix, uint64_t n_rows, uint64_t seed);
/* The Gaussian-mixture corpus of SURVEY.md §8(d) ("1000 centres, sigma = 0.1", the shape of cmd/kmeans-test-data's
 * clusters mode, main.go:231-283), generated ON DEVICE: row r = centre[hash(r) % n_centres] + sigma * N(0,1) per element,
 * centres U[-1,1)^dim.  unit_norm != 0 follows the reference tool to the letter (unit-length centres, rows normalised after
 * the noise).  The near-tie stress case of the filter paths; device-only generator — tests read the rows back. */
int nk_index_fill_clustered(NkIndex *ix, uint64_t n_rows, uint64_t seed, uint32_t n_centres, float sigma, int unit_norm);
/* Single-device index only: this process owns rows [row_base, row_base+n) of a larger corpus
 * (multi-process sharding, one rank per GPU).  Emitted indices are global.  Also offsets the synthetic
 * generator so rank g's rows equal rows row_base.. of the global stream. */
int nk_index_set_row_base(NkIndex *ix, uint64_t row_base);
/* Adopt caller-owned device memory as the (single) shard; not freed by nk_index_release.  The rows may still change behind
 * the library's back (the reference normalises its buffer right after creating it, gpu.go:2100-2106), so no BF16 shadow is
 * built until the caller says the rows are final: nk_index_refresh_shadow. */
int nk_index_attach_device_rows(NkIndex *ix, void *rows_dev, uint64_t n_rows);
/* (Re)build the 16-bit image the fast filter path streams (BF16 shadow + norms of fp32 rows; |x|^2 of fp16 / bf16 rows) from
 * the rows as they are NOW.  For attached rows this is what gives the documented drop-in route (INTEGRATION.md step 2) the
 * headline path; call it again whenever the caller rewrites its buffer. */
int nk_index_refresh_shadow(NkIndex *ix);
/* Change the metric of subsequent searches (rows are stored raw and the shadow is metric-independent: nothing is rebuilt). */
int nk_index_set_metric(NkIndex *ix, int metric);
/* Score floor of subsequent searches, evaluated INSIDE the kernels (it seeds every query's running threshold, so it also
 * prunes): cosine / dot — rows scoring below min_score are never returned (VectorIndex.Search minSimilarity,
 * vector_index.go:339-352; queryNodes keeps a node only if bestScore >= 0, call_vector.go:243); euclidean — the value is a
 * MAXIMUM distance.  Queries with fewer than k admissible rows return 0xffffffff / 0 in the unused slots.  -INFINITY
 * (euclidean: +INFINITY or any negative value) clears it. */
int nk_index_set_min_score(NkIndex *ix, float min_score);
int nk_index_set_path(NkIndex *ix, int path);
uint64_t nk_index_rows(const NkIndex *ix);
int nk_index_stats(const NkIndex *ix, NkStats *out);
/* Diagnostics: copies the device status words of shard 0 after synchronising: out[0] = candidate-buffer overflow
 * (always 0 in a correct run), out[1] != 0 if the last filter stage overflowed its margin buffers and the exact kernels
 * queued behind it produced the result, out[2] = bit pattern of max |x|^2 seen by that search, out[3] = 1 if the BF16
 * shadow stage overflowed and the TF32 filter over the fp32 rows re-ran the search. */
int nk_index_debug_flags(NkIndex *ix, int out[4]);
/* Cumulative diagnostics of shard 0: out[0] = filter searches whose first (16-bit) stage overflowed its margin buffers and
 * re-ran through the TF32 filter, out[1] = filter searches that fell through to the exact kernels, out[2] = longest
 * per-query survivor list of the last filter search, out[3] = OR of the overflow reasons seen so far (1 = a margin buffer
 * could not be pruned below its refill mark, 2 = a CTA's emission was cut at its slot count, 8 = non-finite bound).
 * (Retry rate of a corpus = out[0..1] / searches.) */
int nk_index_debug_counters(NkIndex *ix, uint64_t out[4]);
/* Tests only: the raw score estimate and the error bound the filter kernels compare with, for EVERY (row, query) pair of
 * a single-device index: est_host / bnd_host are [rows x Q] floats (row-major, Q <= 64).  which = NK_PATH_TENSOR_FILTER
 * (1xTF32 pass over fp32 rows) or NK_PATH_TENSOR_SHADOW (16-bit pass).  The filters are sound iff |est - exact| <= bnd;
 * tests/test_gpu_error_model.py measures the worst err / bnd ratio against fp64 on adversarial data. */
int nk_debug_filter_dump(NkIndex *ix, const float *queries_host, uint32_t Q, int which, float *est_host, float *bnd_host);
/* Device-resident searches return before the device has run: this waits for `stream` (and the index's own streams), reads
 * and clears the sticky internal-overflow word nk_search checks on every call, and returns 0 / -1 with that message. */
int nk_index_status(NkIndex *ix, void *stream);
/* Which kernel the last search used: NK_PATH_SIMT / _TENSOR / _TENSOR_FILTER / _TENSOR_SHADOW (-1: null index). */
int nk_index_last_path(const NkIndex *ix);
/* Device-side timing of the dominant kernel (bench.py roofline): when enabled, the main scan launches of
 * every search (CUDA-core or tensor-core scan; query prep and list merge excluded) are bracketed by CUDA
 * events on their stream.  nk_index_scan_time_ms synchronises, returns the summed duration and the number
 * of main scan launches since the last call, and resets the counters. */
int nk_index_enable_timing(NkIndex *ix, int enabled);
int nk_index_scan_time_ms(NkIndex *ix, double *total_ms, uint64_t *scan_launches);
/* Copy n_rows rows starting at global row `row` back to the host (tests / Serialize). */
int nk_index_read_rows(NkIndex *ix, uint64_t row, uint64_t n_rows, void *rows_host);

/* Batched fused search.  queries_host: [Q x dim] fp32.  out_idx/out_score: caller-owned [Q x k]
 * (row stride k).  Returns the number of results per query, min(k, N) (cuda_bridge.go:647-649;
 * 0 for k == 0 or an empty index, cuda_bridge.go:644-646, gpu.go:1540-1542), or -1 on error.
 * Order: cosine/dot — score descending, ties by row index ascending; euclidean — distance ascending,
 * ties by row index ascending, out_score = the distance (callers apply 1/(1+d), similarity.go:152-158).
 * Synchronous: inputs are consumed and outputs complete on return. */
int nk_search(NkIndex *ix, const float *queries_host, uint32_t Q, uint32_t k, uint32_t *out_idx, float *out_score);

/* Same, single-device index, everything device-resident and asynchronous on `stream` (a cudaStream_t,
 * NULL = the index's own stream).  queries_dev [Q x dim] fp32; out_idx_dev/out_score_dev [Q x k]. */
int nk_search_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t *out_idx_dev,
                     float *out_score_dev, void *stream);

/* Multi-process sharding (one rank per GPU): emit this shard's sorted candidate list as packed 64-bit
 * keys [Q x k] (order-preserving score bits << 32 | ~row index; larger key = better), to be exchanged
 * (e.g. ncclAllGather of Q*k*8 bytes per rank) and merged with nk_merge_keys_device. */
int nk_search_keys_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint64_t *out_keys_dev,
                          void *stream);
/* Merge n_lists candidate lists laid out [n_lists][Q][k] into final [Q x k] idx/score on the current
 * device of `device_id`.  metric selects the score decoding (euclidean: distance).  With a stream the call is
 * asynchronous on it (the searches that produced the keys must be ordered before it on that stream); with
 * stream == NULL it synchronises the device first and returns after the merge has completed. */
int nk_merge_keys_device(int device_id, const uint64_t *keys_dev, uint32_t n_lists, uint32_t Q, uint32_t k,
                         int metric, uint32_t *out_idx_dev, float *out_score_dev, void *stream);

/* Best-of-chunks per node — the scoring loop of db.index.vector.queryNodes (call_vector.go:177-256) on the device.  Rows are
 * chunk embeddings; group_of_row[r] in [0, n_groups) is the node row r belongs to (host array, one entry per row; NULL
 * clears; cleared by row-count changing mutations like the row mask).  nk_search_groups scores ONE query against every
 * admissible row (row mask = label filter, score floor = "bestScore >= 0"), keeps each node's best chunk with a per-node
 * atomic max (segment-max) and returns the k best nodes: out_group / out_row / out_score [k] = node id, row of its best
 * chunk, that chunk's score (euclidean: distance), ordered by (score desc, row asc).  Returns the number of nodes found.
 * Exact fp32 arithmetic, no over-select loop.  Single-device indexes. */
int nk_index_set_row_groups(NkIndex *ix, const uint32_t *group_of_row, uint64_t n_rows, uint32_t n_groups);
int nk_search_groups(NkIndex *ix, const float *query_host, uint32_t k, uint32_t *out_group, uint32_t *out_row, float *out_score);

/* Cluster-routed search (ClusterIndex.SearchWithClusters, pkg/gpu/kmeans.go:816-836), single-device indexes.
 * nk_index_set_clusters installs a clustering: K <= NK_MAX_CLUSTERS centroids [K x dim] fp32 (host) and one assignment per row
 * (host int32 [n_rows], n_rows == rows of the index); entries outside [0, K) put the row in no cluster; centroids == NULL
 * clears.  The device keeps the centroids and the members sorted by (cluster, row) (built on the device, rows are read in
 * place).  Cleared by every row-count changing mutation (upload / append / remove_swap / fill / attach), like the row groups;
 * update_row keeps it (the new contents are scored, the assignment is the caller's business).
 * nk_search_clusters answers Q queries at once.  Per query: route to the P = min(n_probe, K) centroids nearest in squared
 * Euclidean distance (float32 differences, float64 squares), nearest first, ties to the lower centroid id (FindNearestClusters,
 * kmeans.go:734-777); score exactly in fp32, with the index's metric, every member of those clusters that the row mask admits,
 * score floor honoured; return the best k, ordered by (score desc | distance asc), ties by position in the candidate list
 * (probe rank, then ascending row: the order GetClusterMembers + SearchCandidates see).  out_idx / out_score [Q x k]; slots
 * beyond a query's candidate count hold 0xffffffff / 0.  out_probe (nullable) [Q x P] = the routed clusters.  Returns
 * min(k, rows of the index) (0 for k == 0, Q == 0 or an empty index) or -1: k > NK_MAX_K, n_probe == 0, several devices,
 * "no clusters set".  Host-synchronous (one synchronisation).  The _device form is asynchronous on `stream` (NULL = the
 * index's own), with device pointers, no host round trip and no allocation per call; overflow of an internal capacity is
 * reported by nk_index_status. */
#define NK_MAX_CLUSTERS 4096u
int nk_index_set_clusters(NkIndex *ix, const float *centroids_host, uint32_t K, const int32_t *assign_host, uint64_t n_rows);
int nk_search_clusters(NkIndex *ix, const float *queries_host, uint32_t Q, uint32_t k, uint32_t n_probe, uint32_t *out_idx,
                       float *out_score, int32_t *out_probe);
int nk_search_clusters_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t n_probe, uint32_t *out_idx_dev,
                              float *out_score_dev, int32_t *out_probe_dev, void *stream);

/* Row-sharded search, one rank per GPU, exchange BEHIND the ABI (SURVEY.md §8e; the reference has a single DeviceID,
 * gpu.go:218).  Each rank owns rows [row_base, row_base + n) (nk_index_set_row_base).  The only data that crosses GPUs is
 * every rank's Q*k candidate keys, pushed with plain peer stores over NVLink into a small buffer each rank exports through
 * CUDA IPC — no NCCL, no host hop, two launches (csrc/exchange.cu):
 *   c = nk_comm_create(device, rank, world, slot_bytes >= max Q*k*8);  nk_comm_export(c, handle[64]);
 *   (the host exchanges the world handles by any transport);  nk_comm_connect(c, all_handles = world x 64 B in rank order);
 *   nk_search_sharded_device(ix, c, queries_dev, Q, k, out_idx_dev, out_score_dev, stream)  on every rank, same sequence.
 * Ranks living in ONE process (several single-device indexes) use nk_comm_connect_local instead of export / connect.
 * nk_comm_status synchronises the stream and reports a peer that never arrived (the device-side wait is bounded: 2 s). */
NkComm *nk_comm_create(int device_id, int rank, int world, size_t slot_bytes);
int nk_comm_export(NkComm *c, void *handle_out);
int nk_comm_connect(NkComm *c, const void *handles);
int nk_comm_connect_local(NkComm **comms, int world);
int nk_comm_status(NkComm *c, void *stream);
void nk_comm_release(NkComm *c);
/* The exchange step alone: keys_dev = this rank's [Q x k] keys (e.g. from nk_search_keys_device, ordered before on
 * `stream`); writes the merged, decoded result. */
int nk_comm_exchange_merge(NkComm *c, const uint64_t *keys_dev, uint32_t Q, uint32_t k, int metric, uint32_t *out_idx_dev,
                           float *out_score_dev, void *stream);
int nk_search_sharded_device(NkIndex *ix, NkComm *comm, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t *out_idx_dev,
                             float *out_score_dev, void *stream);

/* Score an explicit subset of rows (global indices) against one query and return them sorted
 * (EmbeddingIndex.ScoreSubset gpu.go:1552-1616, ClusterIndex.SearchCandidates kmeans.go:839-895).
 * out arrays have length min(k, n_rows_subset) per query; returns that length or -1. */
int nk_score_subset(NkIndex *ix, const float *query_host, const uint32_t *rows_host, uint32_t n_subset, uint32_t k,
                    uint32_t *out_idx, float *out_score);

/* k-means routing on device (pkg/gpu/kmeans.go, SURVEY.md §8(f)4) for fp32 indexes.
 * nk_index_assign_nearest = assignToCentroids (kmeans.go:458-489, metric NK_METRIC_EUCLIDEAN: nearest by squared
 * distance) / assignToCentroidsGPU (kmeans.go:491-546, NK_METRIC_COSINE: highest cosine): the fused scan with the roles
 * swapped — the K centroids (host, [K x dim]) are the corpus, the index's rows are the queries, read in place.
 * assign_io (host, [rows], int32) holds the previous assignment on entry (any value, e.g. 0 as in Go) and the new one
 * on return; *changed (nullable) = how many differ.  Ties go to the lowest centroid index.
 * nk_index_cluster_means = updateCentroidsWithBuffer (kmeans.go:585-618): centroids_io (host, [K x dim]) <- float32 of the
 * float64 mean of each cluster's rows; clusters without members keep their value; counts_out (nullable, [K]). */
int nk_index_assign_nearest(NkIndex *ix, const float *centroids_host, uint32_t K, int metric, int32_t *assign_io,
                            uint64_t *changed);
int nk_index_cluster_means(NkIndex *ix, const int32_t *assign_host, uint32_t K, float *centroids_io, uint32_t *counts_out);
/* k-means++ seeding (initCentroidsKMeansPlusPlus, kmeans.go:364-427) over every row of an fp32 index, on the device.
 * Centroid 0 = row first_row.  For c = 1 .. K-1: D2[i] = min over chosen centroids of squaredEuclidean(row i, centroid)
 * (float32 differences, float64 squares); target = draws[c-1] * sum(D2) in float64; centroid c = the first row i with
 * cumsum(D2)[0..i] >= target, or the last row when there is none (NaN total).  A row whose distance to the new centroid
 * is not strictly smaller keeps its D2 (strict <, kmeans.go:414-421).  draws (host, [K-1], values in [0, 1)) are the
 * caller's uniform variates (rand.Float64), so the result is reproducible.  centroids_out (host, [K x dim]) = those
 * rows; rows_out (nullable, [K]) = their row positions in the index (first_row's numbering, across all shards);
 * rows_scored (nullable) = how many (row, step) distances were computed rather than skipped by the triangle-inequality
 * bound.  Every row takes part, and the row mask is not consulted (like nk_index_assign_nearest).  Multi-device indexes
 * are supported.  Returns 0, or -1 for: a non-fp32 index, K == 0, K > rows, first_row >= rows, or draws == NULL with
 * K > 1. */
int nk_index_kmeanspp(NkIndex *ix, uint32_t K, uint64_t first_row, const double *draws, float *centroids_out,
                      uint32_t *rows_out, uint64_t *rows_scored);

/* Synthetic fp32 query block from the shared generator, on the device of a single-device index. */
int nk_fill_uniform_device(int device_id, float *out_dev, uint64_t n_rows, uint32_t dim, uint64_t seed,
                           uint64_t row_base, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* NORNIC_KNN_H */
