// kernels.cuh — internal launcher interface between the C-ABI host code and the kernels.
#pragma once
#include <utility>
#include <vector>

#include "common.cuh"

namespace nk {

struct DeviceInfo {
    int device_id = 0;
    int num_sms = 148;
    size_t max_smem_optin = 0;
    int cc = 0;
};
int query_device_info(int device_id, DeviceInfo *out);

// Grow-only device scratch of one shard (never freed between searches: no per-query cudaMalloc,
// unlike cuda.Device.Search, cuda_bridge.go:652-663).
struct Workspace {
    uint64_t *cand = nullptr;     size_t cand_bytes = 0;     // [grid][QT][cap] candidate buffers
    uint64_t *partial = nullptr;  size_t partial_bytes = 0;  // [Q][grid][k] per-CTA sorted lists
    uint64_t *keys = nullptr;     size_t keys_bytes = 0;     // [Q][k] merged keys
    uint64_t *below = nullptr;    size_t below_bytes = 0;    // [Q] exclusion bounds of the k > NK_MAX_K passes
    uint64_t *keys2 = nullptr;    size_t keys2_bytes = 0;    // filter mode: shared thresholds gtau[] + list fills gcount[]; big-k: per-pass keys
    float *queries = nullptr;     size_t queries_bytes = 0;  // staged queries (host API)
    uint32_t *out_idx = nullptr;  size_t out_idx_bytes = 0;
    float *out_score = nullptr;   size_t out_score_bytes = 0;
    float *qaux = nullptr;        size_t qaux_bytes = 0;     // tensor path: split / normalised queries
    float *rownorm = nullptr;     size_t rownorm_bytes = 0;  // tensor path: per-row inverse norms / sq norms
    int *flags = nullptr;   // NK_FLAG_WORDS ints of device status (layout: FLAG_* in scan_tensor_shared.cuh)
    uint32_t *sub_rows = nullptr; size_t sub_rows_bytes = 0;  // nk_score_subset: row ids + gathered rows (no per-call alloc)
    void *sub_gather = nullptr;   size_t sub_gather_bytes = 0;
    void *scratch = nullptr;      size_t scratch_bytes = 0;    // k-means routing / group search scratch
    // cached TMA descriptors (tc_cached_map): re-encoded only when the base pointer or shape changes
    struct MapSlot {
        alignas(64) unsigned char bytes[128];
        uint64_t key[6];
        bool valid = false;
    };
    MapSlot maps[8];
    int release();
};
int ws_reserve(void **p, size_t *cur, size_t need);

struct ScanArgs {
    const void *rows = nullptr;  // [n x dim] row-major, fp32 or fp16
    int dtype = NK_DTYPE_F32;
    uint32_t n = 0;
    uint32_t dim = 0;
    uint64_t row_base = 0;       // global index of row 0
    const float *queries = nullptr;  // device [Q x dim] fp32
    uint32_t Q = 0;
    uint32_t k = 0;              // 1..NK_MAX_K (may exceed n: missing slots are key 0)
    int metric = NK_METRIC_COSINE;
    cudaStream_t stream = nullptr;
    // optional timing of the dominant kernel only (bench roofline): events recorded on `stream` right before the
    // first and right after the last main scan launch (query prep / list merge excluded); *main_launches += count
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    uint64_t *main_launches = nullptr;
    const int *only_if = nullptr;  // CUDA-core scan as a device-side conditional fallback (runs only if *only_if != 0)
    // k > NK_MAX_K is served by repeated passes: pass p only admits keys strictly below below[q] (the last key the
    // previous pass returned for query q); nullptr = no bound.  CUDA-core scan only.
    const uint64_t *below = nullptr;
    // optional row filter (label / tombstone bitmask): bit r (LSB first in 32-bit words) set = local row r takes part;
    // nullptr = every row.  Honoured by every scan kernel.
    const uint32_t *row_mask = nullptr;
    // optional BF16 shadow of an fp32 shard (scan_tensor_shadow.cu): rows of `shadow_dimpad` bf16 + per-row |x|^2 and
    // |x - bf16(x)|^2; nullptr = none
    const void *shadow = nullptr;
    uint32_t shadow_dimpad = 0;
    bool shadow_native = false;  // 16-bit corpus: shadow == rows (row stride dim * 2 bytes), dnorm2 == nullptr
    const float *xnorm2 = nullptr, *dnorm2 = nullptr;
    // optional fused decode: the final (index, score) arrays [Q x k] are written by the last kernel of the path
    uint32_t *out_idx = nullptr;
    float *out_score = nullptr;
    // caller's score floor in key space (cosine / dot: similarity; euclidean: -distance^2): lower-scoring rows are never
    // returned (VectorIndex.Search minSimilarity, vector_index.go:339-352; queryNodes bestScore >= 0, call_vector.go:243)
    float min_score = -INFINITY;
    // filter paths: do not queue the retry / exact stages; the (host-synchronous) caller inspects the status words and
    // calls scan_tensor_filter_tail only when a stage overflowed
    bool defer_tail = false;
};

// Fused distance + top-k scan on CUDA cores (small Q, any dim / dtype / alignment).
// Writes per-query sorted candidate keys [Q][k] to out_keys (device).
int scan_simt(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, uint64_t *out_keys, uint64_t *launches);

// Merge n_lists sorted (or unsorted) key lists per query into the best k, sorted descending.
// key(list l, query q, slot i) = keys[l*list_stride + q*q_stride + i], i < list_len (0 = k).
// only_if != nullptr: the kernel returns at once unless *only_if != 0 (device-side conditional fallback).
// dec_idx / dec_score != nullptr: also write the decoded (index, score) arrays [Q x k] (fused decode_keys; dec_metric).
// q_lists != nullptr (device [Q]): query q merges only its first q_lists[q] <= n_lists lists.
int merge_keys(const uint64_t *keys, uint32_t n_lists, size_t list_stride, size_t q_stride, uint32_t Q, uint32_t k,
               uint64_t *out_keys, cudaStream_t stream, const int *only_if = nullptr, uint32_t list_len = 0,
               uint32_t *dec_idx = nullptr, float *dec_score = nullptr, int dec_metric = 0, const uint32_t *wait_flags = nullptr,
               uint32_t wait_epoch = 0, int *wait_err = nullptr, const uint32_t *q_lists = nullptr);
// keys [Q][k] -> idx/score [Q][k]; euclidean decodes score = sqrt(-s).
int decode_keys(const uint64_t *keys, uint32_t Q, uint32_t k, int metric, uint32_t *out_idx, float *out_score,
                cudaStream_t stream, const int *only_if = nullptr);

// Row utilities (legacy ABI + index maintenance).
int row_norms(const float *rows, float *norms, uint32_t n, uint32_t dim, cudaStream_t s);
int normalize_rows(float *rows, uint32_t n, uint32_t dim, cudaStream_t s);
int row_scores(const float *rows, const float *query, float *scores, uint32_t n, uint32_t dim, int normalized,
               cudaStream_t s);
int topk_scores(const DeviceInfo &di, const float *scores, uint32_t n, uint32_t k, Workspace &ws, uint64_t *out_keys,
                cudaStream_t s, const uint64_t *below = nullptr);
// below[q] = keys[q*k + k-1] (the smallest key pass p returned): the exclusion bound of pass p+1.
int update_below(const uint64_t *keys, uint32_t Q, uint32_t k, uint64_t *below, cudaStream_t s);
int fill_uniform(void *out, int dtype, uint64_t n_rows, uint32_t dim, uint64_t seed, uint64_t row_base, cudaStream_t s);
int fill_clustered(void *out, int dtype, uint64_t n_rows, uint32_t dim, uint64_t seed, uint64_t row_base, uint32_t centres, float sigma,
                   int unit, cudaStream_t s);
// |x|^2 of rows [first, first+count) of an fp16 / bf16 corpus -> out[first..]
int row_sqnorms16(const void *rows, int dtype, uint64_t first, uint64_t count, uint32_t dim, float *out, cudaStream_t s);
// best-of-chunks per node (queryNodes): best[group[r]] = max key over the node's rows; top-k over the node keys; decode
int group_best(const void *rows, int dtype, uint64_t n, uint32_t dim, uint64_t row_base, const float *query, int metric,
               const uint32_t *group, const uint32_t *mask, float min_score, unsigned long long *best, cudaStream_t s);
int topk_keys(const DeviceInfo &di, const unsigned long long *keys, uint32_t n, uint32_t k, Workspace &ws, uint64_t *out_keys,
              cudaStream_t s);
int decode_group_keys(const uint64_t *keys, uint32_t k, int metric, const uint32_t *group, uint64_t row_base, uint32_t *out_group,
                      uint32_t *out_row, float *out_score, cudaStream_t s);
// k-means update step on device (kmeans.go:585-618): fp64 per-cluster sums + member counts (the K x dim means are
// finished on the host); count_changed = |{i : a[i] != b[i]}| accumulated into *changed.
int cluster_sums(const float *rows, uint64_t n, uint32_t dim, const int32_t *assign, uint32_t K, double *sums,
                 unsigned long long *counts, cudaStream_t s);
int count_changed(const int32_t *a, const uint32_t *b, uint64_t n, unsigned long long *changed, cudaStream_t s);

// ---- k-means++ seeding (kmeanspp.cu) --------------------------------------------------------------------------------------
// Per shard: d2 [n] fp64 (distance to the nearest chosen centroid), near [n] (its index), bsum [ceil(n / KPP_BLOCK)] fp64
// block sums of d2, cen [K x dim] the chosen centroids, cc [K] fp64 distances from the newest centroid to the earlier ones.
constexpr uint32_t KPP_BLOCK = 1024;  // rows per fixed partial-sum block
// d2 <- min(d2, squaredEuclidean(row, cen[c])) (strict <), skipping rows the triangle-inequality bound rules out; init:
// d2 <- squaredEuclidean(row, cen[0]) for every row.  Rewrites bsum; *scored += rows whose distance was computed.
int kpp_update(const DeviceInfo &di, const float *rows, uint64_t n, uint32_t dim, const float *cen, uint32_t c, bool init,
               const double *cc, double *d2, int32_t *near, double *bsum, unsigned long long *scored, cudaStream_t s);
// Selection of centroid c, one CTA.  mode KPP_SELECT: target = draws[c-1] * total, copies the chosen row into cen[c] and
// its local id into sel[c] (n - 1 when no row reaches the target).  KPP_TOTAL: *total_out = sum of bsum.  KPP_SELECT_AT:
// the given target and offset of this shard, *pick_out = the chosen local row or -1 when none reaches the target.
enum { KPP_SELECT = 0, KPP_TOTAL = 1, KPP_SELECT_AT = 2 };
int kpp_select(int mode, const double *d2, const double *bsum, uint64_t n, const double *draws, uint32_t c, double target,
               double offset, const float *rows, uint32_t dim, float *cen, uint32_t *sel, double *total_out, long long *pick_out,
               cudaStream_t s);
// cc[j] = sqrt(squaredEuclidean(cen[c], cen[j])) for j < c.
int kpp_cc(const float *cen, uint32_t c, uint32_t dim, double *cc, cudaStream_t s);
int convert_f32_to_16(const float *src, void *dst, int dtype, size_t n, cudaStream_t s);  // fp16 / bf16, round to nearest even like the host's astype
int gather_rows(const void *rows, int dtype, uint32_t dim, const uint32_t *idx, uint32_t n_idx, void *out,
                cudaStream_t s);

// ---- cluster-routed search (cluster_search.cu) ----------------------------------------------------------------------------
// Device layout of an installed clustering: centroids [K x dim], CSR offsets [K+1] and member rows (local ids) sorted by
// (cluster, row).  Rows assigned outside [0, K) belong to no cluster.  Host copies of the sizes the planner needs.
struct ClusterLayout {
    float *centroids = nullptr;   size_t centroids_bytes = 0;
    uint32_t *offs = nullptr;     size_t offs_bytes = 0;
    uint32_t *members = nullptr;  size_t members_bytes = 0;
    void *build = nullptr;        size_t build_bytes = 0;  // counting-sort scratch (per-tile histograms, assignments)
    uint32_t K = 0, max_rows = 0;
    uint64_t n_assigned = 0;
    bool on = false;
    void release();
};
int cluster_layout_build(ClusterLayout &L, const float *centroids_host, uint32_t K, uint32_t dim, const int32_t *assign_host,
                         uint64_t n_rows, cudaStream_t s, uint64_t *launches);

// Grow-only scratch of the routed search: one arena carved per call, plus the route kernel's per-query-group arrival
// counters (zero between calls: the last CTA of a group resets its own).
struct ClusterSearchWs {
    void *arena = nullptr;      size_t arena_bytes = 0;
    int *counters = nullptr;    size_t counters_bytes = 0;
    uint64_t *cand = nullptr;   size_t cand_bytes = 0;
    int release();
};
struct ClusterSearchArgs {
    const void *rows = nullptr;
    int dtype = NK_DTYPE_F32;
    uint32_t dim = 0;
    uint64_t row_base = 0;
    const uint32_t *row_mask = nullptr;
    float min_score = -INFINITY;  // key space
    int metric = NK_METRIC_COSINE;
    const float *queries = nullptr;  // device [Q x dim]
    uint32_t Q = 0, k = 0, n_probe = 0;
    uint32_t *out_idx = nullptr;  // device [Q x k]
    float *out_score = nullptr;
    int32_t *out_probe = nullptr;  // device [Q x min(n_probe, K)] or nullptr
    int *flags = nullptr;
    cudaStream_t stream = nullptr;
    bool timing = false;  // record an event pair around every scan launch into *timing_events
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> *timing_events = nullptr;
};
int cluster_search(const DeviceInfo &di, const ClusterLayout &L, const ClusterSearchArgs &a, ClusterSearchWs &ws, uint64_t *launches);

}  // namespace nk
