// index_api.cu — the fused batched kNN API (Part 2 of include/nornic_knn.h).
//
// NkIndex is the device-side half of gpu.EmbeddingIndex (pkg/gpu/gpu.go:1224-1260): a flat row-major
// [N x dim] corpus resident in HBM, row-sharded by contiguous ranges over the GPUs of this process.
// nk_search replaces cuda.Device.Search (pkg/gpu/cuda/cuda_bridge.go:643-686: NewBuffer + NewEmptyBuffer
// + CosineSimilarity + TopK, with a cudaMalloc/cudaFree pair and an n-float D2H per query) by one
// fused scan per shard + a candidate merge; nothing is allocated per query and only Q*k results leave
// the device.
#include <algorithm>
#include <map>
#include <mutex>
#include <stdlib.h>
#include <string.h>
#include <thread>
#include <vector>

#include "kernels.cuh"
#include "scan_tensor_shared.cuh"

namespace nk {
int scan_tensor(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, uint64_t *out_keys, uint64_t *launches);
bool scan_tensor_supported(const DeviceInfo &di, const ScanArgs &a);
int scan_tensor_filter(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, uint64_t *out_keys, uint64_t *launches);
int scan_tensor_filter_tail(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, uint64_t *out_keys, uint64_t *launches);
int scan_filter_dump(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, int which, float *est, float *bnd, uint32_t ld, uint64_t *launches);
bool scan_tensor_filter_supported(const DeviceInfo &di, const ScanArgs &a);
bool shadow_pass_supported(const DeviceInfo &di, const ScanArgs &a);
bool assign_tensor_supported(const DeviceInfo &di, uint32_t dim, uint32_t K, int metric);
int assign_tensor(const DeviceInfo &di, const float *rows, const void *shadow, uint32_t dimpad, const float *xnorm2, const float *dnorm2,
                  uint32_t n, uint32_t dim, const float *centroids_dev, uint32_t K, int metric, uint32_t *assign_dev, cudaStream_t stream,
                  uint64_t *launches, void **scratch, size_t *scratch_bytes);
int build_shadow(const float *rows, uint64_t first, uint64_t count, uint32_t dim, uint32_t dimpad, void *shadow, float *xnorm2,
                 float *dnorm2, cudaStream_t stream);
}

struct NkShard {
    int device = 0;
    nk::DeviceInfo di;
    cudaStream_t stream = nullptr;
    void *rows = nullptr;
    bool owns = true;
    uint64_t n = 0, cap = 0, base = 0;
    // BF16 shadow of an owned fp32 shard (scan_tensor_shadow.cu): rows [0, shadow_n) are converted; capacity in rows
    // 16-bit shards (fp16 / bf16) are scanned in place by the same kernel: they only carry xnorm2 (shadow stays null).
    void *shadow = nullptr;
    float *xnorm2 = nullptr, *dnorm2 = nullptr;
    uint64_t shadow_cap = 0, shadow_n = 0;
    bool shadow_attached = false;  // caller-owned rows: shadow built on request (nk_index_refresh_shadow)
    // last filter search (host-synchronous API): what the deferred retry tail needs
    nk::ScanArgs last_args;
    uint64_t *last_out_keys = nullptr;
    bool last_filter = false;
    uint32_t *group = nullptr;  // node id per row (nk_index_set_row_groups), local rows
    size_t group_bytes = 0;
    bool group_on = false;
    nk::ClusterLayout clusters;  // nk_index_set_clusters (single-device indexes)
    nk::ClusterSearchWs cws;
    nk::Workspace ws;
    uint64_t *h_keys = nullptr;  // pinned staging for multi-shard host merge
    size_t h_keys_bytes = 0;
    unsigned char *h_res = nullptr;  // pinned staging of a single-shard result: [idx][score][status words] in ONE sync
    size_t h_res_bytes = 0;
    // cold-start feed: two pinned staging buffers + their "copy drained" events (stream_h2d)
    void *stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_ev[2] = {nullptr, nullptr};
    void *cvt = nullptr;  // device scratch for fp32 -> fp16 conversion at load
    uint32_t *mask = nullptr;  // optional row filter (nk_index_set_row_mask): bit = local row
    size_t mask_bytes = 0;
    bool mask_on = false;
    size_t cvt_bytes = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timing;  // pending scan-kernel event pairs
    std::vector<uint64_t> timing_launches;
};

struct NkIndex {
    uint32_t dim = 0;
    int dtype = NK_DTYPE_F32;
    int metric = NK_METRIC_COSINE;
    int path = NK_PATH_AUTO;
    bool shadow_on = true;  // NK_SHADOW=0 at creation: never build the BF16 shadow (saves 50% HBM, halves filter speed)
    bool timing_on = false;
    int last_path = NK_PATH_SIMT;
    uint64_t row_base = 0;
    std::vector<NkShard> shards;
    uint64_t mask_alive = 0;  // rows that pass the row mask (all shards); meaningful while a mask is set
    bool mask_on = false;
    float min_score = -INFINITY;  // score floor of subsequent searches, in the API's score domain (nk_index_set_min_score)
    uint32_t n_groups = 0;        // nk_index_set_row_groups
    NkStats stats{};
    std::mutex mu;
    size_t esz() const { return dtype == NK_DTYPE_F32 ? 4 : 2; }
    // the floor in key space: euclidean keys are -distance^2 and the API's floor is a maximum distance
    float key_floor() const {
        if (metric == NK_METRIC_EUCLIDEAN) return (min_score >= 0.0f && min_score < INFINITY) ? -(min_score * min_score) : -INFINITY;
        return min_score > -INFINITY ? min_score : -INFINITY;
    }
    uint32_t dimpad() const { return (dim + 63) / 64 * 64; }
    uint64_t rows() const {
        uint64_t t = 0;
        for (auto &s : shards) t += s.n;
        return t;
    }
};

// Row-count changing mutations invalidate the row mask (its bits are positions), the row groups and the clustering.
static void drop_row_mask(NkIndex *ix) {
    ix->mask_on = false;
    ix->n_groups = 0;
    for (auto &s : ix->shards) { s.mask_on = false; s.group_on = false; s.clusters.on = false; }
}

static void shard_drop_shadow(NkShard &s) {
    if (s.shadow) cudaFree(s.shadow);
    if (s.xnorm2) cudaFree(s.xnorm2);
    if (s.dnorm2) cudaFree(s.dnorm2);
    s.shadow = nullptr; s.xnorm2 = s.dnorm2 = nullptr;
    s.shadow_cap = s.shadow_n = 0;
}

// Bring the 16-bit image of a shard up to date with rows [0, s.n) (converting only what is missing): the BF16 shadow + norms
// of an fp32 shard, or just the |x|^2 array of an fp16 / bf16 shard (scanned in place).  It is an optimisation: if its memory
// cannot be had the shard simply goes without (TF32 filter / CUDA-core scan over the rows).
static int shard_sync_shadow(NkIndex *ix, NkShard &s) {
    const bool f32 = ix->dtype == NK_DTYPE_F32;
    const bool wanted = ix->shadow_on && (s.owns || s.shadow_attached) && ix->dim >= 32 && s.n > 0 && (f32 ? ix->dim % 4 == 0 : ix->dim % 8 == 0);
    if (!wanted) {
        s.shadow_n = 0;
        return 0;
    }
    const uint32_t dimpad = ix->dimpad();
    if (s.shadow_cap < s.n) {
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        shard_drop_shadow(s);
        const uint64_t cap = s.cap > s.n ? s.cap : s.n;
        cudaError_t e = f32 ? cudaMalloc(&s.shadow, cap * dimpad * 2) : cudaSuccess;
        if (e == cudaSuccess) e = cudaMalloc((void **)&s.xnorm2, cap * 4);
        if (e == cudaSuccess && f32) e = cudaMalloc((void **)&s.dnorm2, cap * 4);
        if (e != cudaSuccess) {
            cudaGetLastError();
            shard_drop_shadow(s);
            return 0;
        }
        s.shadow_cap = cap;
    }
    if (s.shadow_n < s.n) {
        if (f32) {
            if (nk::build_shadow(static_cast<const float *>(s.rows), s.shadow_n, s.n - s.shadow_n, ix->dim, dimpad, s.shadow, s.xnorm2,
                                 s.dnorm2, s.stream))
                return -1;
        } else if (nk::row_sqnorms16(s.rows, ix->dtype, s.shadow_n, s.n - s.shadow_n, ix->dim, s.xnorm2, s.stream)) {
            return -1;
        }
        ix->stats.kernel_launches++;
    }
    s.shadow_n = s.n;
    return 0;
}
static int shard_shadow_row(NkIndex *ix, NkShard &s, uint64_t local) {  // one row changed in place
    if (!s.xnorm2 || local >= s.shadow_n) return 0;
    ix->stats.kernel_launches++;
    if (ix->dtype != NK_DTYPE_F32) return nk::row_sqnorms16(s.rows, ix->dtype, local, 1, ix->dim, s.xnorm2, s.stream);
    return nk::build_shadow(static_cast<const float *>(s.rows), local, 1, ix->dim, ix->dimpad(), s.shadow, s.xnorm2, s.dnorm2, s.stream);
}

// ---- cold-start feed (SURVEY.md §8(f)3) ---------------------------------------------------------------------------
// Host rows -> device through two pinned staging buffers: while chunk i crosses PCIe by DMA the CPU copies chunk i+1
// into the other buffer, so pageable (and unaligned: the vectors of a serialized index start at an arbitrary byte
// offset) sources load at the slower of the host memcpy and the PCIe rate instead of the driver's pageable path.
// cvt_f32_to_f16: the source is fp32 and the destination rows are fp16 (down-conversion at load, on the device).
constexpr size_t STAGE_BYTES = 32u << 20;

// one core copies ~11 GB/s, a x16 Gen5 link moves ~50: split the staging copy over a few threads
static void parallel_memcpy(void *dst, const void *src, size_t bytes) {
    constexpr int T = 6;
    if (bytes < (4u << 20)) {
        memcpy(dst, src, bytes);
        return;
    }
    std::thread th[T - 1];
    const size_t part = (bytes / T + 63) & ~(size_t)63;
    for (int t = 1; t < T; ++t) {
        const size_t lo = std::min(bytes, part * t), hi = t == T - 1 ? bytes : std::min(bytes, part * (t + 1));
        th[t - 1] = std::thread([=] { if (hi > lo) memcpy(static_cast<char *>(dst) + lo, static_cast<const char *>(src) + lo, hi - lo); });
    }
    memcpy(dst, src, std::min(bytes, part));
    for (auto &t : th) t.join();
}

static int stream_h2d(NkShard &s, void *dst_dev, const void *src_host, size_t bytes, bool cvt_f32_to_f16 = false, int cvt_dtype = NK_DTYPE_F16) {
    if (bytes == 0) return 0;
    for (int i = 0; i < 2; ++i) {
        if (!s.stage[i]) NK_CUDA_OK(cudaHostAlloc(&s.stage[i], STAGE_BYTES, cudaHostAllocDefault));
        if (!s.stage_ev[i]) NK_CUDA_OK(cudaEventCreateWithFlags(&s.stage_ev[i], cudaEventDisableTiming));
    }
    if (cvt_f32_to_f16 && nk::ws_reserve(&s.cvt, &s.cvt_bytes, 2 * STAGE_BYTES)) return -1;
    size_t done = 0;
    for (int i = 0; done < bytes; ++i) {
        const int b = i & 1;
        const size_t chunk = std::min(STAGE_BYTES, bytes - done);
        if (i >= 2) NK_CUDA_OK(cudaEventSynchronize(s.stage_ev[b]));  // the DMA that last read this buffer has drained
        parallel_memcpy(s.stage[b], static_cast<const char *>(src_host) + done, chunk);
        if (cvt_f32_to_f16) {
            float *scratch = reinterpret_cast<float *>(static_cast<char *>(s.cvt) + (size_t)b * STAGE_BYTES);
            NK_CUDA_OK(cudaMemcpyAsync(scratch, s.stage[b], chunk, cudaMemcpyHostToDevice, s.stream));
            if (nk::convert_f32_to_16(scratch, static_cast<char *>(dst_dev) + done / 2, cvt_dtype, chunk / 4, s.stream)) return -1;
        } else {
            NK_CUDA_OK(cudaMemcpyAsync(static_cast<char *>(dst_dev) + done, s.stage[b], chunk, cudaMemcpyHostToDevice, s.stream));
        }
        NK_CUDA_OK(cudaEventRecord(s.stage_ev[b], s.stream));
        done += chunk;
    }
    return 0;
}

static int shard_reserve_rows(NkIndex *ix, NkShard &s, uint64_t need_rows, bool keep) {
    if (need_rows <= s.cap && s.rows) return 0;
    if (!s.owns) {
        nk::set_error("cannot grow attached (caller-owned) device rows");
        return -1;
    }
    uint64_t cap = keep ? std::max<uint64_t>(need_rows, s.cap + s.cap / 2) : need_rows;
    if (cap < 16) cap = 16;
    void *p = nullptr;
    size_t rb = (size_t)ix->dim * ix->esz();
    NK_CUDA_OK(cudaMalloc(&p, cap * rb));
    if (s.rows) {
        if (keep && s.n) NK_CUDA_OK(cudaMemcpyAsync(p, s.rows, s.n * rb, cudaMemcpyDeviceToDevice, s.stream));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        NK_CUDA_OK(cudaFree(s.rows));
    }
    s.rows = p;
    s.cap = cap;
    return 0;
}

static void rebase(NkIndex *ix) {
    uint64_t b = ix->row_base;
    for (auto &s : ix->shards) {
        s.base = b;
        b += s.n;
    }
    ix->stats.rows = ix->rows();
}

// Locate the shard holding global row `row` (relative to row_base).
static NkShard *find_shard(NkIndex *ix, uint64_t row, uint64_t *local) {
    for (auto &s : ix->shards)
        if (row >= s.base - ix->row_base && row < s.base - ix->row_base + s.n) {
            *local = row - (s.base - ix->row_base);
            return &s;
        }
    return nullptr;
}

struct ScanOut {  // optional extras of run_scan
    uint32_t *out_idx = nullptr;   // fused decode (single-shard searches)
    float *out_score = nullptr;
    bool defer_tail = false;       // host-synchronous caller: retry stages are queued only if a flag was raised
};
static int run_scan(NkIndex *ix, NkShard &s, const float *q_dev, uint32_t Q, uint32_t k, uint64_t *out_keys,
                    cudaStream_t stream, const ScanOut &xo = ScanOut());

// k > NK_MAX_K (the reference accepts any k, cuda_bridge.go:327-375): ceil(k / NK_MAX_K) fused CUDA-core passes; pass p+1
// only admits keys strictly below the last key pass p returned, so the passes tile the ranking exactly.
static int run_scan_bigk(NkIndex *ix, NkShard &s, const float *q_dev, uint32_t Q, uint32_t k, uint64_t *out_keys,
                         cudaStream_t stream, const void *rows = nullptr, uint32_t n_rows = 0, bool custom_rows = false) {
    if (nk::ws_reserve((void **)&s.ws.below, &s.ws.below_bytes, (size_t)Q * 8)) return -1;
    if (nk::ws_reserve((void **)&s.ws.keys2, &s.ws.keys2_bytes, (size_t)Q * NK_MAX_K * 8)) return -1;
    NK_CUDA_OK(cudaMemsetAsync(s.ws.below, 0xff, (size_t)Q * 8, stream));
    for (uint32_t done = 0; done < k;) {
        const uint32_t kp = k - done < NK_MAX_K ? k - done : NK_MAX_K;
        nk::ScanArgs a;
        a.rows = custom_rows ? rows : s.rows; a.dtype = ix->dtype; a.n = custom_rows ? n_rows : (uint32_t)s.n; a.dim = ix->dim;
        a.row_base = custom_rows ? 0 : s.base;
        a.queries = q_dev; a.Q = Q; a.k = kp; a.metric = ix->metric; a.stream = stream; a.below = s.ws.below;
        a.row_mask = (!custom_rows && s.mask_on) ? s.mask : nullptr;
        a.min_score = custom_rows ? -INFINITY : ix->key_floor();
        if (nk::scan_simt(s.di, a, s.ws, s.ws.keys2, &ix->stats.kernel_launches)) return -1;
        NK_CUDA_OK(cudaMemcpy2DAsync(out_keys + done, (size_t)k * 8, s.ws.keys2, (size_t)kp * 8, (size_t)kp * 8, Q,
                                     cudaMemcpyDeviceToDevice, stream));
        if (nk::update_below(s.ws.keys2, Q, kp, s.ws.below, stream)) return -1;
        ix->stats.kernel_launches++;
        ix->stats.bytes_scanned += (uint64_t)s.n * ix->dim * ix->esz() * ((Q + 7) / 8);
        done += kp;
    }
    ix->last_path = NK_PATH_SIMT;
    return 0;
}

static int run_scan(NkIndex *ix, NkShard &s, const float *q_dev, uint32_t Q, uint32_t k, uint64_t *out_keys,
                    cudaStream_t stream, const ScanOut &xo) {
    s.last_filter = false;
    if (k > NK_MAX_K) {
        if (run_scan_bigk(ix, s, q_dev, Q, k, out_keys, stream)) return -1;
        if (xo.out_idx) {
            if (nk::decode_keys(out_keys, Q, k, ix->metric, xo.out_idx, xo.out_score, stream)) return -1;
            ix->stats.kernel_launches++;
        }
        return 0;
    }
    nk::ScanArgs a;
    a.rows = s.rows; a.dtype = ix->dtype; a.n = (uint32_t)s.n; a.dim = ix->dim; a.row_base = s.base;
    a.queries = q_dev; a.Q = Q; a.k = k; a.metric = ix->metric; a.stream = stream;
    a.row_mask = s.mask_on ? s.mask : nullptr;
    a.out_idx = xo.out_idx; a.out_score = xo.out_score; a.min_score = ix->key_floor(); a.defer_tail = xo.defer_tail;
    // AUTO (measured on B200, N=10M d=1024, ms per batch).  fp32 rows: CUDA-core scan 5.9 / 6.2 / 6.1 / 7.6 at Q = 1 / 2 /
    // 4 / 8, TF32 tensor filter 5.8 for any Q <= 64 -> CUDA cores keep Q <= 4, tensor cores from 5 queries on.  With a
    // BF16 shadow the filter streams half the bytes: 2.9-3.1 ms for any Q <= 128, so it serves every batch size once the
    // shard is large enough for bytes (not launches) to matter; small shards keep the single-kernel CUDA-core scan at
    // Q <= 4 (N=100k d=128: 86 us vs 89 us).  16-bit shards: the 16-bit tensor pass from 5 queries on (the CUDA-core scan
    // already streams the minimum bytes at Q <= 4).
    nk::ScanArgs as = a;  // with the 16-bit image attached (if the shard has an up-to-date one)
    if (s.xnorm2 && s.shadow_n == s.n) {
        if (ix->dtype == NK_DTYPE_F32) {
            as.shadow = s.shadow; as.dnorm2 = s.dnorm2;
        } else {
            as.shadow = s.rows; as.shadow_native = true;
        }
        as.shadow_dimpad = ix->dimpad(); as.xnorm2 = s.xnorm2;
    }
    const bool tensor_ok = nk::scan_tensor_supported(s.di, a);
    const bool filter_ok = ix->dtype == NK_DTYPE_F32 && nk::scan_tensor_filter_supported(s.di, a);
    const bool shadow_ok = as.shadow != nullptr && nk::shadow_pass_supported(s.di, as) && nk::scan_tensor_filter_supported(s.di, as);
    int use = NK_PATH_SIMT;
    if (ix->path == NK_PATH_TENSOR || ix->path == NK_PATH_TENSOR_FILTER || ix->path == NK_PATH_TENSOR_SHADOW) {
        if (!(ix->path == NK_PATH_TENSOR ? tensor_ok : ix->path == NK_PATH_TENSOR_FILTER ? filter_ok : shadow_ok)) {
            nk::set_error("tensor path %d does not support this shape (dim=%u dtype=%d metric=%d Q=%u k=%u shadow=%d)", ix->path, ix->dim,
                          ix->dtype, ix->metric, Q, k, (int)(as.shadow != nullptr));
            return -1;
        }
        use = ix->path;
    } else if (ix->path == NK_PATH_AUTO) {
        const bool big_shard = (uint64_t)s.n * ix->dim * 4 >= (64ull << 20);
        if (Q >= 5) use = shadow_ok ? NK_PATH_TENSOR_SHADOW : filter_ok ? NK_PATH_TENSOR_FILTER : tensor_ok ? NK_PATH_TENSOR : NK_PATH_SIMT;
        else if (shadow_ok && big_shard && ix->dtype == NK_DTYPE_F32) use = NK_PATH_TENSOR_SHADOW;
    }
    if (use == NK_PATH_TENSOR_SHADOW) a = as;
    const bool use_tensor = use != NK_PATH_SIMT;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    uint64_t main_launches = 0;
    if (ix->timing_on) {
        NK_CUDA_OK(cudaEventCreate(&e0));
        NK_CUDA_OK(cudaEventCreate(&e1));
        a.ev_begin = e0; a.ev_end = e1; a.main_launches = &main_launches;
    }
    const bool is_filter = use == NK_PATH_TENSOR_FILTER || use == NK_PATH_TENSOR_SHADOW;
    NK_RANGE_PUSH(use == NK_PATH_TENSOR_SHADOW ? "nk:scan:shadow" : use == NK_PATH_TENSOR_FILTER ? "nk:scan:tf32-filter"
                  : use == NK_PATH_TENSOR ? "nk:scan:3xtf32" : "nk:scan:simt");
    int rc = is_filter ? nk::scan_tensor_filter(s.di, a, s.ws, out_keys, &ix->stats.kernel_launches)
             : use == NK_PATH_TENSOR ? nk::scan_tensor(s.di, a, s.ws, out_keys, &ix->stats.kernel_launches)
                                     : nk::scan_simt(s.di, a, s.ws, out_keys, &ix->stats.kernel_launches);
    NK_RANGE_POP();
    if (ix->timing_on) {
        if (rc == 0 && main_launches) {
            s.timing.emplace_back(e0, e1);
            s.timing_launches.push_back(main_launches);
        } else {
            cudaEventDestroy(e0);
            cudaEventDestroy(e1);
        }
    }
    ix->last_path = use;
    if (rc == 0 && is_filter) {
        s.last_filter = true;
        s.last_args = a;
        s.last_args.ev_begin = s.last_args.ev_end = nullptr;
        s.last_args.main_launches = nullptr;
        s.last_out_keys = out_keys;
    }
    if (rc == 0)
        ix->stats.bytes_scanned += use == NK_PATH_TENSOR_SHADOW ? (uint64_t)s.n * (ix->dtype == NK_DTYPE_F32 ? ix->dimpad() : ix->dim) * 2 * ((Q + 127) / 128)
                                   : (uint64_t)s.n * ix->dim * ix->esz() * (use == NK_PATH_TENSOR_FILTER ? ((Q + 127) / 128) : use_tensor ? ((Q + 63) / 64) : ((Q + 7) / 8));
    return rc;
}

// Host-synchronous searches defer the retry / exact stages of the filter paths: after the stream has drained, look at the
// status words; only if a stage overflowed (adversarial near-ties, NaN rows) queue the tail, wait again and let the caller
// re-read the results.  Returns 1 if a retry ran, 0 if not, -1 on error (a fatal candidate-buffer overflow included).
static int finish_deferred(NkIndex *ix, NkShard &s) {
    int h[nk::NK_FLAG_WORDS];
    NK_CUDA_OK(cudaMemcpyAsync(h, s.ws.flags, sizeof(h), cudaMemcpyDeviceToHost, s.stream));
    NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    int retried = 0;
    if (s.last_filter && s.last_args.defer_tail && (h[nk::FLAG_RETRY] || h[nk::FLAG_OVERFLOW])) {
        NK_RANGE_PUSH("nk:retry-tail");
        const int rc = nk::scan_tensor_filter_tail(s.di, s.last_args, s.ws, s.last_out_keys, &ix->stats.kernel_launches);
        NK_RANGE_POP();
        if (rc) return -1;
        NK_CUDA_OK(cudaMemcpyAsync(h, s.ws.flags, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        retried = 1;
    }
    s.last_filter = false;
    if (h[nk::FLAG_FATAL]) {
        cudaMemsetAsync(s.ws.flags, 0, sizeof(int), s.stream);
        nk::set_error("internal: candidate buffer overflow (flag=%d)", h[nk::FLAG_FATAL]);
        return -1;
    }
    return retried;
}

extern "C" {

const char *nk_last_error(void) { return nk::get_error(); }
const char *nk_version(void) { return "nornic-knn-b200 0.1 (sm_100a)"; }

NkIndex *nk_index_create(const int *device_ids, int n_devices, uint32_t dim, int dtype, int metric) {
    nk::DeviceGuard _restore_device;
    if (n_devices <= 0 || !device_ids || dim == 0) {
        nk::set_error("nk_index_create: need >= 1 device and dim > 0");
        return nullptr;
    }
    if (dtype != NK_DTYPE_F32 && dtype != NK_DTYPE_F16 && dtype != NK_DTYPE_BF16) {
        nk::set_error("nk_index_create: unknown dtype %d", dtype);
        return nullptr;
    }
    if (metric < NK_METRIC_COSINE || metric > NK_METRIC_EUCLIDEAN) {
        nk::set_error("nk_index_create: unknown metric %d", metric);
        return nullptr;
    }
    NkIndex *ix = new NkIndex();
    ix->dim = dim; ix->dtype = dtype; ix->metric = metric;
    if (const char *e = getenv("NK_SHADOW")) ix->shadow_on = atoi(e) != 0;  // read once, at creation
    ix->stats.dim = dim; ix->stats.n_devices = (uint32_t)n_devices;
    ix->shards.resize(n_devices);
    for (int i = 0; i < n_devices; ++i) {
        NkShard &s = ix->shards[i];
        s.device = device_ids[i];
        cudaError_t e = cudaSetDevice(s.device);
        if (e == cudaSuccess && nk::query_device_info(s.device, &s.di) != 0) e = cudaErrorUnknown;
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaMalloc((void **)&s.ws.flags, sizeof(int) * nk::NK_FLAG_WORDS);
        if (e == cudaSuccess) e = cudaMemset(s.ws.flags, 0, sizeof(int) * nk::NK_FLAG_WORDS);
        if (e != cudaSuccess) {
            if (e != cudaErrorUnknown) nk::set_error("nk_index_create(device %d): %s", s.device, cudaGetErrorString(e));
            cudaGetLastError();
            nk_index_release(ix);
            return nullptr;
        }
    }
    return ix;
}

void nk_index_release(NkIndex *ix) {
    nk::DeviceGuard _restore_device;
    if (!ix) return;
    for (auto &s : ix->shards) {
        cudaSetDevice(s.device);
        if (s.stream) {
            cudaStreamSynchronize(s.stream);
            cudaStreamDestroy(s.stream);
        }
        if (s.rows && s.owns) cudaFree(s.rows);
        shard_drop_shadow(s);
        if (s.h_keys) cudaFreeHost(s.h_keys);
        if (s.h_res) cudaFreeHost(s.h_res);
        for (int i = 0; i < 2; ++i) {
            if (s.stage[i]) cudaFreeHost(s.stage[i]);
            if (s.stage_ev[i]) cudaEventDestroy(s.stage_ev[i]);
        }
        if (s.cvt) cudaFree(s.cvt);
        if (s.mask) cudaFree(s.mask);
        if (s.group) cudaFree(s.group);
        s.clusters.release();
        s.cws.release();
        s.ws.release();
    }
    delete ix;
}

static int upload_impl(NkIndex *ix, const void *rows_host, uint64_t n_rows, bool src_is_f32) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    if (n_rows && !rows_host) { nk::set_error("null rows"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    drop_row_mask(ix);
    const bool cvt = src_is_f32 && ix->dtype != NK_DTYPE_F32;
    const size_t rb = (size_t)ix->dim * ix->esz(), src_rb = (size_t)ix->dim * (cvt ? 4 : ix->esz());
    const uint64_t G = ix->shards.size();
    // global row ids are 32-bit on this boundary (SearchResult.Index uint32, cuda_bridge.go:425-428)
    if (ix->row_base + n_rows > 0xfffffff0ull) { nk::set_error("index exceeds 2^32 rows (row ids are uint32)"); return -1; }
    uint64_t off = 0;
    for (uint64_t g = 0; g < G; ++g) {
        NkShard &s = ix->shards[g];
        uint64_t cnt = n_rows * (g + 1) / G - n_rows * g / G;  // contiguous range [g*N/G, (g+1)*N/G)
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (!s.owns) { s.rows = nullptr; s.owns = true; s.cap = 0; s.shadow_attached = false; }
        s.n = 0;
        if (shard_reserve_rows(ix, s, cnt, false)) return -1;
        if (stream_h2d(s, s.rows, static_cast<const char *>(rows_host) + off * src_rb, cnt * src_rb, cvt, ix->dtype)) return -1;
        s.n = cnt;
        s.shadow_n = 0;
        if (shard_sync_shadow(ix, s)) return -1;
        off += cnt;
        ix->stats.bytes_h2d += cnt * src_rb;
    }
    for (auto &s : ix->shards) {
        NK_CUDA_OK(cudaSetDevice(s.device));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    }
    rebase(ix);
    (void)rb;
    return 0;
}

int nk_index_upload(NkIndex *ix, const void *rows_host, uint64_t n_rows) { return upload_impl(ix, rows_host, n_rows, false); }

int nk_index_upload_from_f32(NkIndex *ix, const float *rows_host_f32, uint64_t n_rows) { return upload_impl(ix, rows_host_f32, n_rows, true); }

// Serialized index (EmbeddingIndex.Serialize, gpu.go:2373-2412): LE [dims u32][count u32][count x (len u32, id bytes)]
// [count x dims fp32].  Walks the id table; the vectors start at *vec_offset (any byte alignment).
int nk_blob_vectors(const void *blob, size_t blob_bytes, uint32_t *dims, uint32_t *count, size_t *vec_offset) {
    if (!blob || !dims || !count || !vec_offset) { nk::set_error("null argument"); return -1; }
    const unsigned char *p = static_cast<const unsigned char *>(blob);
    auto rd32 = [&](size_t at) { return (uint32_t)p[at] | ((uint32_t)p[at + 1] << 8) | ((uint32_t)p[at + 2] << 16) | ((uint32_t)p[at + 3] << 24); };
    if (blob_bytes < 8) { nk::set_error("gpu: invalid serialized data"); return -1; }  // gpu.go:2419-2421
    const uint32_t d = rd32(0), c = rd32(4);
    size_t off = 8;
    for (uint32_t i = 0; i < c; ++i) {
        if (off + 4 > blob_bytes) { nk::set_error("serialized index truncated in the id table (id %u)", i); return -1; }
        const uint32_t len = rd32(off);
        off += 4;
        if (len > blob_bytes - off) { nk::set_error("serialized index truncated in the id table (id %u)", i); return -1; }
        off += len;
    }
    if ((uint64_t)c * d * 4 > blob_bytes - off) { nk::set_error("serialized index truncated: %u x %u vectors do not fit", c, d); return -1; }
    *dims = d; *count = c; *vec_offset = off;
    return 0;
}

int nk_index_append(NkIndex *ix, const void *rows_host, uint64_t n_rows) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    if (n_rows == 0) return 0;
    if (!rows_host) { nk::set_error("null rows"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    drop_row_mask(ix);
    NkShard &s = ix->shards.back();
    const size_t rb = (size_t)ix->dim * ix->esz();
    if (ix->row_base + ix->rows() + n_rows > 0xfffffff0ull) { nk::set_error("index exceeds 2^32 rows (row ids are uint32)"); return -1; }
    NK_CUDA_OK(cudaSetDevice(s.device));
    if (shard_reserve_rows(ix, s, s.n + n_rows, true)) return -1;
    if (stream_h2d(s, (char *)s.rows + s.n * rb, rows_host, n_rows * rb)) return -1;
    s.n += n_rows;
    if (shard_sync_shadow(ix, s)) return -1;  // converts only the appended rows (all of them if the shard was regrown)
    NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    ix->stats.bytes_h2d += n_rows * rb;
    rebase(ix);
    return 0;
}

int nk_index_update_row(NkIndex *ix, uint64_t row, const void *row_host) {
    nk::DeviceGuard _restore_device;
    if (!ix || !row_host) { nk::set_error("null argument"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    uint64_t local;
    NkShard *s = find_shard(ix, row, &local);
    if (!s) { nk::set_error("row %llu out of range", (unsigned long long)row); return -1; }
    const size_t rb = (size_t)ix->dim * ix->esz();
    NK_CUDA_OK(cudaSetDevice(s->device));
    NK_CUDA_OK(cudaMemcpyAsync((char *)s->rows + local * rb, row_host, rb, cudaMemcpyHostToDevice, s->stream));
    if (shard_shadow_row(ix, *s, local)) return -1;
    NK_CUDA_OK(cudaStreamSynchronize(s->stream));
    ix->stats.bytes_h2d += rb;
    return 0;
}

int nk_index_remove_swap(NkIndex *ix, uint64_t row) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    uint64_t total = ix->rows();
    if (row >= total) { nk::set_error("row %llu out of range", (unsigned long long)row); return -1; }
    drop_row_mask(ix);
    // last non-empty shard holds the last row
    NkShard *last = nullptr;
    for (auto it = ix->shards.rbegin(); it != ix->shards.rend(); ++it)
        if (it->n) { last = &*it; break; }
    uint64_t local;
    NkShard *s = find_shard(ix, row, &local);
    const size_t rb = (size_t)ix->dim * ix->esz();
    if (row != total - 1) {
        const char *src = (const char *)last->rows + (last->n - 1) * rb;
        char *dst = (char *)s->rows + local * rb;
        // The copy must be ordered with the shard's own stream (non-blocking streams do not synchronise with the legacy
        // default stream): drain the source shard first when it is another device, then copy ON s->stream so that the
        // shadow / norm rebuild queued behind reads the new row.
        if (last != s) {
            NK_CUDA_OK(cudaSetDevice(last->device));
            NK_CUDA_OK(cudaStreamSynchronize(last->stream));
        }
        NK_CUDA_OK(cudaSetDevice(s->device));
        if (last->device == s->device) NK_CUDA_OK(cudaMemcpyAsync(dst, src, rb, cudaMemcpyDeviceToDevice, s->stream));
        else NK_CUDA_OK(cudaMemcpyPeerAsync(dst, s->device, src, last->device, rb, s->stream));
        if (shard_shadow_row(ix, *s, local)) return -1;
        NK_CUDA_OK(cudaStreamSynchronize(s->stream));
    }
    last->n -= 1;
    if (last->shadow_n > last->n) last->shadow_n = last->n;
    rebase(ix);
    return 0;
}

static int fill_impl(NkIndex *ix, uint64_t n_rows, uint64_t seed, uint32_t centres, float sigma, int unit) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    drop_row_mask(ix);
    const uint64_t G = ix->shards.size();
    if (ix->row_base + n_rows > 0xfffffff0ull) { nk::set_error("index exceeds 2^32 rows (row ids are uint32)"); return -1; }
    uint64_t off = 0;
    for (uint64_t g = 0; g < G; ++g) {
        NkShard &s = ix->shards[g];
        uint64_t cnt = n_rows * (g + 1) / G - n_rows * g / G;
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (!s.owns) { s.rows = nullptr; s.owns = true; s.cap = 0; s.shadow_attached = false; }
        s.n = 0;
        if (shard_reserve_rows(ix, s, cnt, false)) return -1;
        if (centres ? nk::fill_clustered(s.rows, ix->dtype, cnt, ix->dim, seed, ix->row_base + off, centres, sigma, unit, s.stream)
                    : nk::fill_uniform(s.rows, ix->dtype, cnt, ix->dim, seed, ix->row_base + off, s.stream))
            return -1;
        ix->stats.kernel_launches++;
        s.n = cnt;
        s.shadow_n = 0;
        if (shard_sync_shadow(ix, s)) return -1;
        off += cnt;
    }
    for (auto &s : ix->shards) {
        NK_CUDA_OK(cudaSetDevice(s.device));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    }
    rebase(ix);
    return 0;
}

int nk_index_fill_uniform(NkIndex *ix, uint64_t n_rows, uint64_t seed) { return fill_impl(ix, n_rows, seed, 0, 0.0f, 0); }
int nk_index_fill_clustered(NkIndex *ix, uint64_t n_rows, uint64_t seed, uint32_t n_centres, float sigma, int unit_norm) {
    if (n_centres == 0) { nk::set_error("nk_index_fill_clustered: n_centres must be >= 1"); return -1; }
    return fill_impl(ix, n_rows, seed, n_centres, sigma, unit_norm);
}

int nk_index_set_row_base(NkIndex *ix, uint64_t row_base) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    if (ix->shards.size() != 1) { nk::set_error("row_base applies to single-device indexes"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->row_base = row_base;
    rebase(ix);
    return 0;
}

int nk_index_attach_device_rows(NkIndex *ix, void *rows_dev, uint64_t n_rows) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    if (ix->shards.size() != 1) { nk::set_error("attach applies to single-device indexes"); return -1; }
    if (ix->row_base + n_rows > 0xfffffff0ull) { nk::set_error("index exceeds 2^32 rows (row ids are uint32)"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    NkShard &s = ix->shards[0];
    NK_CUDA_OK(cudaSetDevice(s.device));
    if (s.rows && s.owns) NK_CUDA_OK(cudaFree(s.rows));
    // caller-owned rows may change behind the library's back (cuda_normalize_vectors runs right after NewBuffer,
    // gpu.go:2100-2106): no shadow until the caller says the rows are final (nk_index_refresh_shadow)
    NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    shard_drop_shadow(s);
    drop_row_mask(ix);
    s.rows = rows_dev; s.owns = false; s.n = n_rows; s.cap = n_rows; s.shadow_attached = false;
    rebase(ix);
    return 0;
}

// (Re)build the 16-bit image of every shard from the rows as they are now.  For attached (caller-owned) rows this is the
// explicit "rows are final" signal that gives the documented drop-in route the fast filter path; for library-owned shards
// it is a no-op unless rows were changed behind the library's back.
int nk_index_refresh_shadow(NkIndex *ix) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    for (auto &s : ix->shards) {
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (!s.owns) s.shadow_attached = true;
        s.shadow_n = 0;
        if (shard_sync_shadow(ix, s)) return -1;
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    }
    return 0;
}

int nk_index_set_metric(NkIndex *ix, int metric) {
    if (!ix) { nk::set_error("null index"); return -1; }
    if (metric < NK_METRIC_COSINE || metric > NK_METRIC_EUCLIDEAN) { nk::set_error("unknown metric %d", metric); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->metric = metric;  // rows are stored raw and the shadow's norms are metric-independent: nothing to rebuild
    return 0;
}

int nk_index_set_min_score(NkIndex *ix, float min_score) {
    if (!ix) { nk::set_error("null index"); return -1; }
    if (min_score != min_score) { nk::set_error("min_score is NaN"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    ix->min_score = min_score;
    return 0;
}

// Row filter for subsequent searches (label / type filter of db.index.vector.queryNodes, call_vector.go:177-193; also
// tombstones): bit r of mask_words (LSB first in 32-bit words) set = row r (relative to the index's first row) may be
// returned.  NULL clears the filter.  Row-count changing mutations (upload, append, remove_swap, fill, attach) clear it.
int nk_index_set_row_mask(NkIndex *ix, const uint32_t *mask_words, uint64_t n_bits) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!mask_words) {  // clear the filter only (the row groups stay: the row count did not change)
        ix->mask_on = false;
        for (auto &s : ix->shards) s.mask_on = false;
        return 0;
    }
    if (n_bits != ix->rows()) { nk::set_error("row mask has %llu bits, index has %llu rows", (unsigned long long)n_bits, (unsigned long long)ix->rows()); return -1; }
    uint64_t off = 0, alive = 0;
    std::vector<uint32_t> local;
    for (auto &s : ix->shards) {
        const size_t words = (size_t)((s.n + 31) / 32);
        local.assign(words ? words : 1, 0u);
        for (uint64_t r = 0; r < s.n; ++r) {
            const uint64_t g = off + r;
            if ((mask_words[g >> 5] >> (g & 31)) & 1u) {
                local[r >> 5] |= 1u << (r & 31);
                ++alive;
            }
        }
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (nk::ws_reserve((void **)&s.mask, &s.mask_bytes, local.size() * 4)) return -1;
        NK_CUDA_OK(cudaMemcpyAsync(s.mask, local.data(), local.size() * 4, cudaMemcpyHostToDevice, s.stream));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        s.mask_on = true;
        off += s.n;
    }
    ix->mask_on = true;
    ix->mask_alive = alive;
    return 0;
}

int nk_index_set_path(NkIndex *ix, int path) {
    if (!ix || path < NK_PATH_AUTO || path > NK_PATH_TENSOR_SHADOW) { nk::set_error("bad path"); return -1; }
    ix->path = path;
    return 0;
}

uint64_t nk_index_rows(const NkIndex *ix) { return ix ? ix->rows() : 0; }

int nk_index_stats(const NkIndex *ix, NkStats *out) {
    if (!ix || !out) { nk::set_error("null argument"); return -1; }
    *out = ix->stats;
    out->rows = ix->rows();
    return 0;
}

int nk_index_debug_flags(NkIndex *ix, int out[4]) {
    nk::DeviceGuard _restore_device;
    if (!ix || !out || ix->shards.empty()) { nk::set_error("null argument"); return -1; }
    NkShard &s = ix->shards[0];
    NK_CUDA_OK(cudaSetDevice(s.device));
    NK_CUDA_OK(cudaDeviceSynchronize());
    int h[nk::NK_FLAG_WORDS];
    NK_CUDA_OK(cudaMemcpy(h, s.ws.flags, sizeof(h), cudaMemcpyDeviceToHost));
    out[0] = h[nk::FLAG_FATAL]; out[1] = h[nk::FLAG_OVERFLOW]; out[2] = h[nk::FLAG_MAXXX]; out[3] = h[nk::FLAG_RETRY];
    return 0;
}

// Cumulative diagnostics of shard 0 since creation: out[0] = filter searches whose first (16-bit) stage overflowed and re-ran
// through the TF32 filter, out[1] = filter searches that fell through to the exact kernels, out[2] = longest per-query
// survivor list of the last filter search.  bench.py reports out[0..1] / searches as the retry rate of a corpus.
int nk_index_debug_counters(NkIndex *ix, uint64_t out[4]) {
    nk::DeviceGuard _restore_device;
    if (!ix || !out || ix->shards.empty()) { nk::set_error("null argument"); return -1; }
    NkShard &s = ix->shards[0];
    NK_CUDA_OK(cudaSetDevice(s.device));
    NK_CUDA_OK(cudaDeviceSynchronize());
    int h[nk::NK_FLAG_WORDS];
    NK_CUDA_OK(cudaMemcpy(h, s.ws.flags, sizeof(h), cudaMemcpyDeviceToHost));
    out[0] = (uint64_t)h[nk::FLAG_N_RETRY]; out[1] = (uint64_t)h[nk::FLAG_N_EXACT]; out[2] = (uint64_t)h[nk::FLAG_LONGEST]; out[3] = (uint64_t)h[nk::FLAG_OVF_BITS];
    return 0;
}

// Tests only: the raw score estimate and the error bound the filter kernels work with, for every (row, query) pair of a
// single-device index (rows x Q floats each, row-major [row][query], host buffers).  which = NK_PATH_TENSOR_FILTER (TF32
// pass over fp32 rows) or NK_PATH_TENSOR_SHADOW (16-bit pass).  The filters are sound iff |est - exact score| <= bnd.
int nk_debug_filter_dump(NkIndex *ix, const float *queries_host, uint32_t Q, int which, float *est_host, float *bnd_host) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (!ix || ix->shards.size() != 1) { nk::set_error("single-device index required"); return -1; }
    s = &ix->shards[0];
    if (!queries_host || !est_host || !bnd_host || Q == 0 || Q > 64 || s->n == 0) { nk::set_error("bad argument (1 <= Q <= 64, non-empty index)"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    NK_CUDA_OK(cudaSetDevice(s->device));
    const size_t cells = (size_t)s->n * Q;
    float *d = nullptr;
    NK_CUDA_OK(cudaMalloc((void **)&d, cells * 8));
    int rc = -1;
    do {
        if (nk::ws_reserve((void **)&s->ws.queries, &s->ws.queries_bytes, (size_t)Q * ix->dim * 4)) break;
        if (cudaMemcpyAsync(s->ws.queries, queries_host, (size_t)Q * ix->dim * 4, cudaMemcpyHostToDevice, s->stream) != cudaSuccess) break;
        if (cudaMemsetAsync(d, 0, cells * 8, s->stream) != cudaSuccess) break;
        nk::ScanArgs a;
        a.rows = s->rows; a.dtype = ix->dtype; a.n = (uint32_t)s->n; a.dim = ix->dim; a.row_base = s->base;
        a.queries = s->ws.queries; a.Q = Q; a.k = 1; a.metric = ix->metric; a.stream = s->stream;
        if (s->xnorm2 && s->shadow_n == s->n) {
            if (ix->dtype == NK_DTYPE_F32) { a.shadow = s->shadow; a.dnorm2 = s->dnorm2; }
            else { a.shadow = s->rows; a.shadow_native = true; }
            a.shadow_dimpad = ix->dimpad(); a.xnorm2 = s->xnorm2;
        }
        if (nk::scan_filter_dump(s->di, a, s->ws, which, d, d + cells, Q, &ix->stats.kernel_launches)) break;
        if (cudaMemcpyAsync(est_host, d, cells * 4, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess) break;
        if (cudaMemcpyAsync(bnd_host, d + cells, cells * 4, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess) break;
        if (cudaStreamSynchronize(s->stream) != cudaSuccess) break;
        rc = 0;
    } while (0);
    if (rc != 0) {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) nk::set_error("nk_debug_filter_dump: %s", cudaGetErrorString(e));
        cudaStreamSynchronize(s->stream);
    }
    cudaFree(d);
    return rc;
}

int nk_index_last_path(const NkIndex *ix) { return ix ? ix->last_path : -1; }

int nk_index_enable_timing(NkIndex *ix, int enabled) {
    if (!ix) { nk::set_error("null index"); return -1; }
    ix->timing_on = enabled != 0;
    return 0;
}

int nk_index_scan_time_ms(NkIndex *ix, double *total_ms, uint64_t *scan_launches) {
    nk::DeviceGuard _restore_device;
    if (!ix || !total_ms || !scan_launches) { nk::set_error("null argument"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    double ms = 0.0;
    uint64_t n = 0;
    for (auto &s : ix->shards) {
        NK_CUDA_OK(cudaSetDevice(s.device));
        for (size_t i = 0; i < s.timing.size(); ++i) {
            float t = 0.0f;
            NK_CUDA_OK(cudaEventSynchronize(s.timing[i].second));
            NK_CUDA_OK(cudaEventElapsedTime(&t, s.timing[i].first, s.timing[i].second));
            ms += t;
            n += s.timing_launches[i];
            cudaEventDestroy(s.timing[i].first);
            cudaEventDestroy(s.timing[i].second);
        }
        s.timing.clear();
        s.timing_launches.clear();
    }
    *total_ms = ms;
    *scan_launches = n;
    return 0;
}

int nk_index_read_rows(NkIndex *ix, uint64_t row, uint64_t n_rows, void *rows_host) {
    nk::DeviceGuard _restore_device;
    if (!ix || (!rows_host && n_rows)) { nk::set_error("null argument"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    const size_t rb = (size_t)ix->dim * ix->esz();
    for (uint64_t i = 0; i < n_rows;) {
        uint64_t local;
        NkShard *s = find_shard(ix, row + i, &local);
        if (!s) { nk::set_error("row %llu out of range", (unsigned long long)(row + i)); return -1; }
        uint64_t cnt = std::min<uint64_t>(n_rows - i, s->n - local);
        NK_CUDA_OK(cudaSetDevice(s->device));
        NK_CUDA_OK(cudaMemcpy((char *)rows_host + i * rb, (const char *)s->rows + local * rb, cnt * rb, cudaMemcpyDeviceToHost));
        ix->stats.bytes_d2h += cnt * rb;
        i += cnt;
    }
    return 0;
}

int nk_search(NkIndex *ix, const float *queries_host, uint32_t Q, uint32_t k, uint32_t *out_idx, float *out_score) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    const uint64_t N = ix->mask_on ? ix->mask_alive : ix->rows();  // rows that can be returned
    if (k == 0 || N == 0 || Q == 0) return 0;  // cuda_bridge.go:644-646, gpu.go:1540-1542
    if (!queries_host || !out_idx || !out_score) { nk::set_error("null argument"); return -1; }
    const uint32_t ke = k > N ? (uint32_t)N : k;  // cuda_bridge.go:647-649
    if (ke > NK_MAX_K_TOTAL) { nk::set_error("k=%u exceeds NK_MAX_K_TOTAL=%u", ke, NK_MAX_K_TOTAL); return -1; }
    const size_t qbytes = (size_t)Q * ix->dim * sizeof(float);
    ix->stats.searches++;
    ix->stats.queries += Q;
    NK_RANGE_PUSH("nk_search");
    struct Pop { ~Pop() { NK_RANGE_POP(); } } pop_on_exit;

    std::vector<NkShard *> live;
    for (auto &s : ix->shards)
        if (s.n) live.push_back(&s);
    const bool single = live.size() == 1;

    // Launch every shard asynchronously, then collect.  A single shard writes the decoded (index, score) arrays from
    // the last kernel of its path (no separate decode launch); the retry stages of the filter paths are deferred.
    for (NkShard *s : live) {
        NK_CUDA_OK(cudaSetDevice(s->device));
        if (nk::ws_reserve((void **)&s->ws.queries, &s->ws.queries_bytes, qbytes)) return -1;
        if (nk::ws_reserve((void **)&s->ws.keys, &s->ws.keys_bytes, (size_t)Q * ke * 8)) return -1;
        ScanOut xo;
        xo.defer_tail = true;
        if (single) {
            if (nk::ws_reserve((void **)&s->ws.out_idx, &s->ws.out_idx_bytes, (size_t)Q * ke * 4)) return -1;
            if (nk::ws_reserve((void **)&s->ws.out_score, &s->ws.out_score_bytes, (size_t)Q * ke * 4)) return -1;
            xo.out_idx = s->ws.out_idx; xo.out_score = s->ws.out_score;
        }
        NK_CUDA_OK(cudaMemcpyAsync(s->ws.queries, queries_host, qbytes, cudaMemcpyHostToDevice, s->stream));
        ix->stats.bytes_h2d += qbytes;
        if (run_scan(ix, *s, s->ws.queries, Q, ke, s->ws.keys, s->stream, xo)) return -1;
    }

    if (single) {
        // Results and status words come back through ONE pinned staging buffer: three short DMA copies and a single stream
        // synchronisation (pageable cudaMemcpyAsync targets cost a driver-side staging round trip each).
        NkShard *s = live[0];
        NK_CUDA_OK(cudaSetDevice(s->device));
        const size_t rbytes = (size_t)Q * ke * 4, need = 2 * rbytes + sizeof(int) * nk::NK_FLAG_WORDS;
        if (s->h_res_bytes < need) {
            if (s->h_res) cudaFreeHost(s->h_res);
            s->h_res = nullptr; s->h_res_bytes = 0;
            NK_CUDA_OK(cudaMallocHost((void **)&s->h_res, need + need / 4));
            s->h_res_bytes = need + need / 4;
        }
        int *hflags = reinterpret_cast<int *>(s->h_res + 2 * rbytes);
        for (int pass = 0; pass < 2; ++pass) {
            NK_CUDA_OK(cudaMemcpyAsync(s->h_res, s->ws.out_idx, rbytes, cudaMemcpyDeviceToHost, s->stream));
            NK_CUDA_OK(cudaMemcpyAsync(s->h_res + rbytes, s->ws.out_score, rbytes, cudaMemcpyDeviceToHost, s->stream));
            NK_CUDA_OK(cudaMemcpyAsync(hflags, s->ws.flags, sizeof(int) * nk::NK_FLAG_WORDS, cudaMemcpyDeviceToHost, s->stream));
            NK_CUDA_OK(cudaStreamSynchronize(s->stream));
            ix->stats.bytes_d2h += (uint64_t)Q * ke * 8;
            if (hflags[nk::FLAG_FATAL]) {
                cudaMemsetAsync(s->ws.flags, 0, sizeof(int), s->stream);
                nk::set_error("internal: candidate buffer overflow (flag=%d)", hflags[nk::FLAG_FATAL]);
                return -1;
            }
            if (pass == 0 && s->last_filter && s->last_args.defer_tail && (hflags[nk::FLAG_RETRY] || hflags[nk::FLAG_OVERFLOW])) {
                // a filter stage overflowed (near-ties, NaN rows): queue the retry / exact stages now and read again
                NK_RANGE_PUSH("nk:retry-tail");
                const int rc = nk::scan_tensor_filter_tail(s->di, s->last_args, s->ws, s->last_out_keys, &ix->stats.kernel_launches);
                NK_RANGE_POP();
                if (rc) return -1;
                continue;
            }
            break;
        }
        s->last_filter = false;
        const uint32_t *hi = reinterpret_cast<const uint32_t *>(s->h_res);
        const float *hs = reinterpret_cast<const float *>(s->h_res + rbytes);
        if (ke == k) {
            memcpy(out_idx, hi, rbytes);
            memcpy(out_score, hs, rbytes);
        } else {
            for (uint32_t q = 0; q < Q; ++q) {
                memcpy(out_idx + (size_t)q * k, hi + (size_t)q * ke, (size_t)ke * 4);
                memcpy(out_score + (size_t)q * k, hs + (size_t)q * ke, (size_t)ke * 4);
            }
        }
        return (int)ke;
    }

    // Multi-shard: gather the per-GPU candidate lists (Q*k*8 B each) and merge on the host with the
    // same (score desc, row asc) order (SURVEY.md §8e "small Q: async D2H + host k-way merge").
    const size_t kbytes = (size_t)Q * ke * 8;
    for (NkShard *s : live) {
        NK_CUDA_OK(cudaSetDevice(s->device));
        if (s->h_keys_bytes < kbytes) {
            if (s->h_keys) cudaFreeHost(s->h_keys);
            s->h_keys = nullptr; s->h_keys_bytes = 0;
            NK_CUDA_OK(cudaMallocHost((void **)&s->h_keys, kbytes + kbytes / 4));
            s->h_keys_bytes = kbytes + kbytes / 4;
        }
    }
    for (NkShard *s : live) {
        NK_CUDA_OK(cudaSetDevice(s->device));
        if (finish_deferred(ix, *s) < 0) return -1;  // runs this shard's retry stages if it needs them
        NK_CUDA_OK(cudaMemcpyAsync(s->h_keys, s->ws.keys, kbytes, cudaMemcpyDeviceToHost, s->stream));
        ix->stats.bytes_d2h += kbytes;
    }
    for (NkShard *s : live) {
        NK_CUDA_OK(cudaSetDevice(s->device));
        NK_CUDA_OK(cudaStreamSynchronize(s->stream));
    }
    std::vector<uint64_t> tmp(live.size() * (size_t)ke);
    for (uint32_t q = 0; q < Q; ++q) {
        size_t m = 0;
        for (NkShard *s : live)
            for (uint32_t i = 0; i < ke; ++i) {
                uint64_t key = s->h_keys[(size_t)q * ke + i];
                if (key) tmp[m++] = key;
            }
        size_t take = std::min<size_t>(ke, m);
        std::partial_sort(tmp.begin(), tmp.begin() + take, tmp.begin() + m, std::greater<uint64_t>());
        for (uint32_t i = 0; i < ke; ++i) {
            if (i < take) {
                float sc = nk::key_score(tmp[i]);
                if (ix->metric == NK_METRIC_EUCLIDEAN) sc = sqrtf(std::max(-sc, 0.0f));
                out_idx[(size_t)q * k + i] = nk::key_row(tmp[i]);
                out_score[(size_t)q * k + i] = sc;
            } else {
                out_idx[(size_t)q * k + i] = 0xffffffffu;
                out_score[(size_t)q * k + i] = 0.0f;
            }
        }
    }
    return (int)ke;
}

static int single_shard(NkIndex *ix, NkShard **out) {
    if (!ix) { nk::set_error("null index"); return -1; }
    if (ix->shards.size() != 1) { nk::set_error("device-resident search needs a single-device index"); return -1; }
    *out = &ix->shards[0];
    return 0;
}

int nk_search_keys_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint64_t *out_keys_dev,
                          void *stream) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    if (k == 0 || Q == 0) return 0;
    if (!queries_dev || !out_keys_dev) { nk::set_error("null argument"); return -1; }
    if (k > NK_MAX_K_TOTAL) { nk::set_error("k=%u exceeds NK_MAX_K_TOTAL=%u", k, NK_MAX_K_TOTAL); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    NK_CUDA_OK(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    ix->stats.searches++;
    ix->stats.queries += Q;
    if (s->n == 0) {
        NK_CUDA_OK(cudaMemsetAsync(out_keys_dev, 0, (size_t)Q * k * 8, st));
        return (int)k;
    }
    if (run_scan(ix, *s, queries_dev, Q, k, out_keys_dev, st)) return -1;
    return (int)k;
}

int nk_search_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t *out_idx_dev,
                     float *out_score_dev, void *stream) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    if (k == 0 || Q == 0) return 0;
    if (!queries_dev || !out_idx_dev || !out_score_dev) { nk::set_error("null argument"); return -1; }
    if (k > NK_MAX_K_TOTAL) { nk::set_error("k=%u exceeds NK_MAX_K_TOTAL=%u", k, NK_MAX_K_TOTAL); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);  // the row count is read under the lock (a concurrent append may change it)
    const uint64_t N = s->n;
    if (N == 0) return 0;
    if (k > N) { nk::set_error("nk_search_device: k=%u > rows=%llu (clamp on the host side)", k, (unsigned long long)N); return -1; }
    NK_CUDA_OK(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (nk::ws_reserve((void **)&s->ws.keys, &s->ws.keys_bytes, (size_t)Q * k * 8)) return -1;
    ix->stats.searches++;
    ix->stats.queries += Q;
    ScanOut xo;
    xo.out_idx = out_idx_dev; xo.out_score = out_score_dev;  // decoded by the last kernel of the path
    if (run_scan(ix, *s, queries_dev, Q, k, s->ws.keys, st, xo)) return -1;
    return (int)k;
}

// Device-resident searches cannot report a (never expected) candidate-buffer overflow when they return: this call waits
// for `stream` (NULL = the index's own streams), reads and clears the sticky status word of every shard, and returns 0 or -1
// with the message nk_search would have given.  Call it wherever the caller synchronises anyway.
int nk_index_status(NkIndex *ix, void *stream) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    int bad = 0;
    for (auto &s : ix->shards) {
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (stream) NK_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        int h = 0;
        NK_CUDA_OK(cudaMemcpy(&h, s.ws.flags, sizeof(int), cudaMemcpyDeviceToHost));
        if (h) {
            NK_CUDA_OK(cudaMemset(s.ws.flags, 0, sizeof(int)));
            bad = h;
        }
    }
    if (bad) { nk::set_error("internal: candidate buffer overflow (flag=%d)", bad); return -1; }
    return 0;
}

// (No scratch buffer: the merge kernel writes the decoded arrays itself, so concurrent merges on different streams share
// nothing.)
int nk_merge_keys_device(int device_id, const uint64_t *keys_dev, uint32_t n_lists, uint32_t Q, uint32_t k, int metric,
                         uint32_t *out_idx_dev, float *out_score_dev, void *stream) {
    nk::DeviceGuard _restore_device;
    if (k == 0 || Q == 0 || n_lists == 0) return 0;
    if (!keys_dev || !out_idx_dev || !out_score_dev) { nk::set_error("null argument"); return -1; }
    if (device_id < 0 || device_id >= 64) { nk::set_error("bad device id %d", device_id); return -1; }
    NK_CUDA_OK(cudaSetDevice(device_id));
    cudaStream_t st = (cudaStream_t)stream;
    // No stream given: behave synchronously (the producers may have run on the indexes' own non-blocking streams,
    // which the legacy default stream does not order against).
    if (!st) NK_CUDA_OK(cudaDeviceSynchronize());
    // one fused launch: merge the lists and write the decoded (index, score) arrays; no intermediate key buffer
    int rc = nk::merge_keys(keys_dev, n_lists, (size_t)Q * k, k, Q, k, nullptr, st, nullptr, 0, out_idx_dev, out_score_dev, metric);
    if (rc == 0 && !st) NK_CUDA_OK(cudaStreamSynchronize(st));
    return rc;
}

int nk_score_subset(NkIndex *ix, const float *query_host, const uint32_t *rows_host, uint32_t n_subset, uint32_t k,
                    uint32_t *out_idx, float *out_score) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    if (n_subset == 0 || k == 0) return 0;
    if (!query_host || !rows_host || !out_idx || !out_score) { nk::set_error("null argument"); return -1; }
    const uint32_t ke = std::min(k, n_subset);
    if (ke > NK_MAX_K_TOTAL) { nk::set_error("k=%u exceeds NK_MAX_K_TOTAL=%u", ke, NK_MAX_K_TOTAL); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    for (uint32_t i = 0; i < n_subset; ++i)
        if (rows_host[i] < ix->row_base || rows_host[i] - ix->row_base >= s->n) {
            nk::set_error("subset row %u out of range", rows_host[i]);
            return -1;
        }
    NK_CUDA_OK(cudaSetDevice(s->device));
    const size_t rb = (size_t)ix->dim * ix->esz();
    // grow-only workspace of the shard: no allocation per call (cuda.Device.Search allocates two buffers per query,
    // cuda_bridge.go:652-663)
    if (nk::ws_reserve((void **)&s->ws.sub_rows, &s->ws.sub_rows_bytes, (size_t)n_subset * 4)) return -1;
    if (nk::ws_reserve(&s->ws.sub_gather, &s->ws.sub_gather_bytes, (size_t)n_subset * rb)) return -1;
    uint32_t *d_rows = s->ws.sub_rows;
    void *d_gather = s->ws.sub_gather;
    std::vector<uint32_t> local(rows_host, rows_host + n_subset);
    for (auto &r : local) r -= (uint32_t)ix->row_base;
    int rc = 0;
    std::vector<uint32_t> pos((size_t)ke);
    do {
        if (cudaMemcpyAsync(d_rows, local.data(), (size_t)n_subset * 4, cudaMemcpyHostToDevice, s->stream) != cudaSuccess) { rc = -1; break; }
        if (nk::gather_rows(s->rows, ix->dtype, ix->dim, d_rows, n_subset, d_gather, s->stream)) { rc = -1; break; }
        if (nk::ws_reserve((void **)&s->ws.queries, &s->ws.queries_bytes, (size_t)ix->dim * 4)) { rc = -1; break; }
        if (nk::ws_reserve((void **)&s->ws.keys, &s->ws.keys_bytes, (size_t)ke * 8)) { rc = -1; break; }
        if (nk::ws_reserve((void **)&s->ws.out_idx, &s->ws.out_idx_bytes, (size_t)ke * 4)) { rc = -1; break; }
        if (nk::ws_reserve((void **)&s->ws.out_score, &s->ws.out_score_bytes, (size_t)ke * 4)) { rc = -1; break; }
        if (cudaMemcpyAsync(s->ws.queries, query_host, (size_t)ix->dim * 4, cudaMemcpyHostToDevice, s->stream) != cudaSuccess) { rc = -1; break; }
        nk::ScanArgs a;
        a.rows = d_gather; a.dtype = ix->dtype; a.n = n_subset; a.dim = ix->dim; a.row_base = 0;
        a.queries = s->ws.queries; a.Q = 1; a.k = ke; a.metric = ix->metric; a.stream = s->stream;
        if (ke > NK_MAX_K) {  // ScoreSubset ranks every candidate (up to MaxCandidates = 5000, vector_pipeline.go:24-31)
            if (run_scan_bigk(ix, *s, s->ws.queries, 1, ke, s->ws.keys, s->stream, d_gather, n_subset, true)) { rc = -1; break; }
            if (nk::decode_keys(s->ws.keys, 1, ke, ix->metric, s->ws.out_idx, s->ws.out_score, s->stream)) { rc = -1; break; }
        } else {
            a.out_idx = s->ws.out_idx; a.out_score = s->ws.out_score;  // decoded by the merge launch
            if (nk::scan_simt(s->di, a, s->ws, s->ws.keys, &ix->stats.kernel_launches)) { rc = -1; break; }
        }
        if (cudaMemcpyAsync(pos.data(), s->ws.out_idx, (size_t)ke * 4, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess) { rc = -1; break; }
        if (cudaMemcpyAsync(out_score, s->ws.out_score, (size_t)ke * 4, cudaMemcpyDeviceToHost, s->stream) != cudaSuccess) { rc = -1; break; }
    } while (0);
    if (rc != 0) {
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) nk::set_error("nk_score_subset: %s", cudaGetErrorString(e));
        cudaStreamSynchronize(s->stream);
        return -1;
    }
    s->last_filter = false;
    if (finish_deferred(ix, *s) < 0) return -1;
    // positions within the subset -> global row ids (ties broken by subset position, like the stable
    // order of ScoreSubset's input list)
    for (uint32_t i = 0; i < ke; ++i) out_idx[i] = pos[i] < n_subset ? rows_host[pos[i]] : 0xffffffffu;
    return (int)ke;
}

// ---- k-means routing on device (pkg/gpu/kmeans.go; SURVEY.md §8(f)4) -----------------------------------------------
// Assignment is the fused scan with the roles swapped: the K centroids are the indexed corpus, the shard's rows are the
// queries — read in place from HBM, 8192 at a time — and k = 1.  Ties go to the lowest centroid index (strict < / >
// in kmeans.go:470-476,529-534).
int nk_index_assign_nearest(NkIndex *ix, const float *centroids_host, uint32_t K, int metric, int32_t *assign_io, uint64_t *changed) {
    nk::DeviceGuard _restore_device;
    if (!ix || !centroids_host || !assign_io) { nk::set_error("null argument"); return -1; }
    if (ix->dtype != NK_DTYPE_F32) { nk::set_error("nk_index_assign_nearest: fp32 index required"); return -1; }
    if (K == 0) { nk::set_error("nk_index_assign_nearest: K must be >= 1"); return -1; }
    if (metric < NK_METRIC_COSINE || metric > NK_METRIC_EUCLIDEAN) { nk::set_error("unknown metric %d", metric); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    uint64_t total_changed = 0, off = 0;
    for (auto &s : ix->shards) {
        if (s.n == 0) continue;
        NK_CUDA_OK(cudaSetDevice(s.device));
        // With a BF16 shadow the assignment is ONE pass of the tensor-core scan with an argmax epilogue (assign_tensor.cu);
        // otherwise the fused kNN scan with the roles swapped: centroids as the corpus, rows as the queries, k = 1.
        const bool tensor = s.shadow && s.shadow_n == s.n && nk::assign_tensor_supported(s.di, ix->dim, K, metric);
        NkIndex *cx = tensor ? nullptr : nk_index_create(&s.device, 1, ix->dim, NK_DTYPE_F32, metric);
        if (!tensor && !cx) return -1;
        // one grow-only scratch buffer per shard, carved up (no cudaMalloc / cudaFree per call)
        const size_t n4 = (s.n * 4 + 255) & ~(size_t)255, cen_b = tensor ? (((size_t)K * ix->dim * 4 + 255) & ~(size_t)255) : 0;
        unsigned long long h_changed = 0;
        int rc = tensor ? 0 : nk_index_upload(cx, centroids_host, K);
        if (rc == 0 && nk::ws_reserve(&s.ws.scratch, &s.ws.scratch_bytes, 3 * n4 + 256 + cen_b)) rc = -1;
        unsigned char *base = static_cast<unsigned char *>(s.ws.scratch);
        uint32_t *d_idx = reinterpret_cast<uint32_t *>(base);
        float *d_sc = reinterpret_cast<float *>(base + n4);
        int32_t *d_prev = reinterpret_cast<int32_t *>(base + 2 * n4);
        unsigned long long *d_changed = reinterpret_cast<unsigned long long *>(base + 3 * n4);
        float *d_cen = reinterpret_cast<float *>(base + 3 * n4 + 256);
        cudaError_t e = cudaSuccess;
        if (rc == 0) {
            if (tensor) e = cudaMemcpyAsync(d_cen, centroids_host, (size_t)K * ix->dim * 4, cudaMemcpyHostToDevice, s.stream);
            if (e == cudaSuccess) e = cudaMemsetAsync(d_changed, 0, 8, s.stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(d_prev, assign_io + off, s.n * 4, cudaMemcpyHostToDevice, s.stream);
            if (e != cudaSuccess) rc = -1;
        }
        if (rc == 0 && tensor) {
            rc = nk::assign_tensor(s.di, static_cast<const float *>(s.rows), s.shadow, ix->dimpad(), s.xnorm2, s.dnorm2, (uint32_t)s.n, ix->dim,
                                   d_cen, K, metric, d_idx, s.stream, &ix->stats.kernel_launches, &s.ws.sub_gather, &s.ws.sub_gather_bytes);
        }
        const uint64_t B = 8192;  // rows per fused search: amortises the ~12 fixed launches of a search over 8 scan launches
        for (uint64_t b = 0; rc == 0 && !tensor && b < s.n; b += B) {
            const uint32_t nb = (uint32_t)std::min<uint64_t>(B, s.n - b);
            if (nk_search_device(cx, static_cast<const float *>(s.rows) + b * ix->dim, nb, 1, d_idx + b, d_sc + b, s.stream) < 0) rc = -1;
        }
        if (rc == 0 && nk::count_changed(d_prev, d_idx, s.n, d_changed, s.stream)) rc = -1;
        if (rc == 0) {
            e = cudaMemcpyAsync(assign_io + off, d_idx, s.n * 4, cudaMemcpyDeviceToHost, s.stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(&h_changed, d_changed, 8, cudaMemcpyDeviceToHost, s.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream);
            if (e != cudaSuccess) rc = -1;
        }
        if (e != cudaSuccess) { nk::set_error("nk_index_assign_nearest: %s", cudaGetErrorString(e)); cudaGetLastError(); }
        cudaStreamSynchronize(s.stream);
        ix->stats.kernel_launches += (cx ? cx->stats.kernel_launches : 0) + 1;
        if (cx) nk_index_release(cx);
        if (rc != 0) return -1;
        total_changed += h_changed;
        off += s.n;
    }
    if (changed) *changed = total_changed;
    return 0;
}

// Update step (kmeans.go:585-618): centroid c <- float32(mean in float64 of the rows assigned to c); clusters without
// members keep their previous position.  Rows with an assignment outside [0, K) are ignored.
int nk_index_cluster_means(NkIndex *ix, const int32_t *assign_host, uint32_t K, float *centroids_io, uint32_t *counts_out) {
    nk::DeviceGuard _restore_device;
    if (!ix || !assign_host || !centroids_io) { nk::set_error("null argument"); return -1; }
    if (ix->dtype != NK_DTYPE_F32) { nk::set_error("nk_index_cluster_means: fp32 index required"); return -1; }
    if (K == 0) return 0;
    std::lock_guard<std::mutex> lk(ix->mu);
    const size_t KD = (size_t)K * ix->dim;
    std::vector<double> sums(KD, 0.0), part(KD);
    std::vector<unsigned long long> counts(K, 0ull), cpart(K);
    uint64_t off = 0;
    for (auto &s : ix->shards) {
        if (s.n == 0) continue;
        NK_CUDA_OK(cudaSetDevice(s.device));
        const size_t kd8 = (KD * 8 + 255) & ~(size_t)255, k8 = ((size_t)K * 8 + 255) & ~(size_t)255;
        if (nk::ws_reserve(&s.ws.scratch, &s.ws.scratch_bytes, kd8 + k8 + s.n * 4)) return -1;  // grow-only, reused across calls
        unsigned char *base = static_cast<unsigned char *>(s.ws.scratch);
        double *d_sums = reinterpret_cast<double *>(base);
        unsigned long long *d_counts = reinterpret_cast<unsigned long long *>(base + kd8);
        int32_t *d_assign = reinterpret_cast<int32_t *>(base + kd8 + k8);
        cudaError_t e = cudaMemsetAsync(d_sums, 0, KD * 8, s.stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(d_counts, 0, (size_t)K * 8, s.stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_assign, assign_host + off, s.n * 4, cudaMemcpyHostToDevice, s.stream);
        int rc = e == cudaSuccess ? nk::cluster_sums(static_cast<const float *>(s.rows), s.n, ix->dim, d_assign, K, d_sums, d_counts, s.stream) : -1;
        if (rc == 0) {
            e = cudaMemcpyAsync(part.data(), d_sums, KD * 8, cudaMemcpyDeviceToHost, s.stream);
            if (e == cudaSuccess) e = cudaMemcpyAsync(cpart.data(), d_counts, (size_t)K * 8, cudaMemcpyDeviceToHost, s.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream);
        }
        if (e != cudaSuccess) { nk::set_error("nk_index_cluster_means: %s", cudaGetErrorString(e)); cudaGetLastError(); rc = -1; }
        cudaStreamSynchronize(s.stream);
        if (rc != 0) return -1;
        ix->stats.kernel_launches++;
        for (size_t i = 0; i < KD; ++i) sums[i] += part[i];
        for (uint32_t c = 0; c < K; ++c) counts[c] += cpart[c];
        off += s.n;
    }
    for (uint32_t c = 0; c < K; ++c) {
        if (counts[c])
            for (uint32_t d = 0; d < ix->dim; ++d) centroids_io[(size_t)c * ix->dim + d] = (float)(sums[(size_t)c * ix->dim + d] / (double)counts[c]);
        if (counts_out) counts_out[c] = (uint32_t)counts[c];
    }
    return 0;
}

// ---- k-means++ seeding on device (initCentroidsKMeansPlusPlus, kmeans.go:364-427; kmeanspp.cu, DESIGN.md §3.8) ---------
// Each shard carves its grow-only scratch into d2 / near / block sums / centroids / cc / draws / picks.  A single-device
// index queues all K - 1 steps on one stream and synchronises once.  A multi-device index picks the shard of each
// selection on the host from the shard totals, summed in shard order; shards are contiguous row ranges, so the global
// cumulative order is the single-device one.  That costs one synchronisation per step.
namespace {
struct KppShard {
    NkShard *s = nullptr;
    uint64_t first = 0;  // index position of the shard's row 0
    double *d2 = nullptr, *bsum = nullptr, *cc = nullptr, *draws = nullptr, *total = nullptr;
    int32_t *near = nullptr;
    float *cen = nullptr;
    uint32_t *sel = nullptr;
    unsigned long long *scored = nullptr;
    long long *pick = nullptr;
};
}  // namespace

static int kmeanspp_steps(NkIndex *ix, std::vector<KppShard> &kv, uint32_t K, uint64_t first_row, const double *draws,
                          float *centroids_out, uint32_t *rows_out, uint64_t *rows_scored) {
    const uint32_t dim = ix->dim;
    const size_t row_bytes = (size_t)dim * 4;
    auto update = [&](KppShard &k, uint32_t c, bool init) {
        ix->stats.kernel_launches++;
        return nk::kpp_update(k.s->di, static_cast<const float *>(k.s->rows), k.s->n, dim, k.cen, c, init, k.cc, k.d2, k.near,
                              k.bsum, k.scored, k.s->stream);
    };
    auto cc = [&](KppShard &k, uint32_t c) {
        ix->stats.kernel_launches++;
        return nk::kpp_cc(k.cen, c, dim, k.cc, k.s->stream);
    };
    std::vector<uint64_t> picked(K, first_row);
    if (kv.size() == 1) {  // every step queued back to back on one stream
        KppShard &k = kv[0];
        NkShard &s = *k.s;
        const float *rows = static_cast<const float *>(s.rows);
        NK_CUDA_OK(cudaSetDevice(s.device));
        if (K > 1) NK_CUDA_OK(cudaMemcpyAsync(k.draws, draws, (size_t)(K - 1) * 8, cudaMemcpyHostToDevice, s.stream));
        NK_CUDA_OK(cudaMemcpyAsync(k.cen, rows + (first_row - k.first) * dim, row_bytes, cudaMemcpyDeviceToDevice, s.stream));
        if (K > 1 && update(k, 0, true)) return -1;
        for (uint32_t c = 1; c < K; ++c) {
            ix->stats.kernel_launches++;
            if (nk::kpp_select(nk::KPP_SELECT, k.d2, k.bsum, s.n, k.draws, c, 0.0, 0.0, rows, dim, k.cen, k.sel, nullptr, nullptr, s.stream))
                return -1;
            if (c + 1 < K && (cc(k, c) || update(k, c, false))) return -1;  // no update after the last selection
        }
        std::vector<uint32_t> sel(K);
        NK_CUDA_OK(cudaMemcpyAsync(centroids_out, k.cen, (size_t)K * row_bytes, cudaMemcpyDeviceToHost, s.stream));
        NK_CUDA_OK(cudaMemcpyAsync(sel.data(), k.sel, (size_t)K * 4, cudaMemcpyDeviceToHost, s.stream));
        NK_CUDA_OK(cudaStreamSynchronize(s.stream));
        for (uint32_t c = 1; c < K; ++c) picked[c] = k.first + sel[c];
    } else {
        // the chosen row travels through the host to every shard's centroid array
        std::vector<float> crow(dim);
        std::vector<double> tot(kv.size());
        auto fetch_row = [&](KppShard &k, uint64_t local) -> int {
            NK_CUDA_OK(cudaSetDevice(k.s->device));
            NK_CUDA_OK(cudaMemcpy(crow.data(), static_cast<const float *>(k.s->rows) + local * dim, row_bytes, cudaMemcpyDeviceToHost));
            return 0;
        };
        auto place = [&](uint32_t c) -> int {
            for (auto &k : kv) {
                NK_CUDA_OK(cudaSetDevice(k.s->device));
                NK_CUDA_OK(cudaMemcpyAsync(k.cen + (size_t)c * dim, crow.data(), row_bytes, cudaMemcpyHostToDevice, k.s->stream));
                if (c + 1 < K && ((c > 0 && cc(k, c)) || update(k, c, c == 0))) return -1;
            }
            return 0;
        };
        for (auto &k : kv)
            if (first_row >= k.first && first_row < k.first + k.s->n && fetch_row(k, first_row - k.first)) return -1;
        if (place(0)) return -1;
        for (uint32_t c = 1; c < K; ++c) {
            for (size_t j = 0; j < kv.size(); ++j) {
                KppShard &k = kv[j];
                NK_CUDA_OK(cudaSetDevice(k.s->device));
                ix->stats.kernel_launches++;
                if (nk::kpp_select(nk::KPP_TOTAL, k.d2, k.bsum, k.s->n, nullptr, c, 0.0, 0.0, nullptr, dim, nullptr, nullptr, k.total,
                                   nullptr, k.s->stream))
                    return -1;
                NK_CUDA_OK(cudaMemcpyAsync(&tot[j], k.total, 8, cudaMemcpyDeviceToHost, k.s->stream));
            }
            double total = 0.0;
            for (size_t j = 0; j < kv.size(); ++j) {
                NK_CUDA_OK(cudaSetDevice(kv[j].s->device));
                NK_CUDA_OK(cudaStreamSynchronize(kv[j].s->stream));
                total += tot[j];
            }
            const double target = draws[c - 1] * total;
            // the first shard whose offset + total reaches the target selects at that offset; one whose in-shard scan
            // falls short by rounding passes on to the next; none (NaN total) -> the last row
            long long pick = -1;
            size_t js = kv.size() - 1;
            double off = 0.0;
            for (size_t j = 0; j < kv.size() && pick < 0; ++j) {
                KppShard &k = kv[j];
                if (off + tot[j] >= target) {
                    NK_CUDA_OK(cudaSetDevice(k.s->device));
                    ix->stats.kernel_launches++;
                    if (nk::kpp_select(nk::KPP_SELECT_AT, k.d2, k.bsum, k.s->n, nullptr, c, target, off, nullptr, dim, nullptr, nullptr,
                                       nullptr, k.pick, k.s->stream))
                        return -1;
                    NK_CUDA_OK(cudaMemcpyAsync(&pick, k.pick, 8, cudaMemcpyDeviceToHost, k.s->stream));
                    NK_CUDA_OK(cudaStreamSynchronize(k.s->stream));
                    if (pick >= 0) js = j;
                }
                off += tot[j];
            }
            const uint64_t local = pick >= 0 ? (uint64_t)pick : kv[js].s->n - 1;
            picked[c] = kv[js].first + local;
            if (fetch_row(kv[js], local) || place(c)) return -1;
        }
        NK_CUDA_OK(cudaSetDevice(kv[0].s->device));
        NK_CUDA_OK(cudaMemcpyAsync(centroids_out, kv[0].cen, (size_t)K * row_bytes, cudaMemcpyDeviceToHost, kv[0].s->stream));
        NK_CUDA_OK(cudaStreamSynchronize(kv[0].s->stream));
    }
    uint64_t scored = 0;
    for (auto &k : kv) {
        unsigned long long v = 0;
        NK_CUDA_OK(cudaSetDevice(k.s->device));
        NK_CUDA_OK(cudaMemcpyAsync(&v, k.scored, 8, cudaMemcpyDeviceToHost, k.s->stream));
        NK_CUDA_OK(cudaStreamSynchronize(k.s->stream));
        scored += v;
    }
    if (rows_scored) *rows_scored = scored;
    if (rows_out)
        for (uint32_t c = 0; c < K; ++c) rows_out[c] = (uint32_t)picked[c];
    ix->stats.bytes_d2h += (uint64_t)K * row_bytes;
    return 0;
}

int nk_index_kmeanspp(NkIndex *ix, uint32_t K, uint64_t first_row, const double *draws, float *centroids_out, uint32_t *rows_out,
                      uint64_t *rows_scored) {
    nk::DeviceGuard _restore_device;
    if (!ix || !centroids_out) { nk::set_error("null argument"); return -1; }
    if (ix->dtype != NK_DTYPE_F32) { nk::set_error("nk_index_kmeanspp: fp32 index required"); return -1; }
    if (K == 0) { nk::set_error("nk_index_kmeanspp: K must be >= 1"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    const uint64_t N = ix->rows();
    if (K > N) { nk::set_error("nk_index_kmeanspp: K=%u exceeds the %llu rows", K, (unsigned long long)N); return -1; }
    if (first_row >= N) { nk::set_error("nk_index_kmeanspp: first_row %llu out of range", (unsigned long long)first_row); return -1; }
    if (K > 1 && !draws) { nk::set_error("nk_index_kmeanspp: K > 1 needs draws"); return -1; }
    NK_RANGE_PUSH("nk_index_kmeanspp");
    struct Pop { ~Pop() { NK_RANGE_POP(); } } pop_on_exit;
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    std::vector<KppShard> kv;
    uint64_t pos = 0;
    for (auto &s : ix->shards) {
        if (s.n == 0) continue;
        NK_CUDA_OK(cudaSetDevice(s.device));
        const uint64_t nblk = (s.n + nk::KPP_BLOCK - 1) / nk::KPP_BLOCK;
        const size_t kd = (size_t)K * ix->dim * 4;
        if (nk::ws_reserve(&s.ws.scratch, &s.ws.scratch_bytes, al(s.n * 8) + al(s.n * 4) + al(nblk * 8) + al(kd) + 2 * al((size_t)K * 8) +
                                                                   al((size_t)K * 4) + 256))
            return -1;
        unsigned char *p = static_cast<unsigned char *>(s.ws.scratch);
        KppShard k;
        k.s = &s;
        k.first = pos;
        k.d2 = reinterpret_cast<double *>(p);          p += al(s.n * 8);
        k.near = reinterpret_cast<int32_t *>(p);       p += al(s.n * 4);
        k.bsum = reinterpret_cast<double *>(p);        p += al(nblk * 8);
        k.cen = reinterpret_cast<float *>(p);          p += al(kd);
        k.cc = reinterpret_cast<double *>(p);          p += al((size_t)K * 8);
        k.draws = reinterpret_cast<double *>(p);       p += al((size_t)K * 8);
        k.sel = reinterpret_cast<uint32_t *>(p);       p += al((size_t)K * 4);
        k.scored = reinterpret_cast<unsigned long long *>(p);
        k.total = reinterpret_cast<double *>(p + 8);
        k.pick = reinterpret_cast<long long *>(p + 16);
        NK_CUDA_OK(cudaMemsetAsync(k.scored, 0, 8, s.stream));
        kv.push_back(k);
        pos += s.n;
    }
    const int rc = kmeanspp_steps(ix, kv, K, first_row, draws, centroids_out, rows_out, rows_scored);
    for (auto &k : kv) {  // nothing stays queued on an error path
        cudaSetDevice(k.s->device);
        cudaStreamSynchronize(k.s->stream);
    }
    if (rc != 0) cudaGetLastError();
    return rc;
}

// ---- best-of-chunks per node (db.index.vector.queryNodes, call_vector.go:177-256; SURVEY.md §8(f)2) -------------------------
// Rows are chunk embeddings; group_of_row[r] = the node row r belongs to (ids in [0, n_groups)).  Stays set until a
// row-count changing mutation (like the row mask, whose bits are positions).
int nk_index_set_row_groups(NkIndex *ix, const uint32_t *group_of_row, uint64_t n_rows, uint32_t n_groups) {
    nk::DeviceGuard _restore_device;
    if (!ix) { nk::set_error("null index"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!group_of_row) {
        ix->n_groups = 0;
        for (auto &s : ix->shards) s.group_on = false;
        return 0;
    }
    if (ix->shards.size() != 1) { nk::set_error("row groups apply to single-device indexes"); return -1; }
    if (n_rows != ix->rows()) { nk::set_error("row groups: %llu entries, index has %llu rows", (unsigned long long)n_rows, (unsigned long long)ix->rows()); return -1; }
    if (n_groups == 0) { nk::set_error("row groups: n_groups must be >= 1"); return -1; }
    for (uint64_t r = 0; r < n_rows; ++r)
        if (group_of_row[r] >= n_groups) { nk::set_error("row groups: group id %u of row %llu out of range", group_of_row[r], (unsigned long long)r); return -1; }
    NkShard &s = ix->shards[0];
    NK_CUDA_OK(cudaSetDevice(s.device));
    if (nk::ws_reserve((void **)&s.group, &s.group_bytes, (size_t)(n_rows ? n_rows : 1) * 4)) return -1;
    NK_CUDA_OK(cudaMemcpyAsync(s.group, group_of_row, n_rows * 4, cudaMemcpyHostToDevice, s.stream));
    NK_CUDA_OK(cudaStreamSynchronize(s.stream));
    s.group_on = true;
    ix->n_groups = n_groups;
    return 0;
}

// One query against the chunk rows; result = the k best NODES, each with the score and row of its best chunk, ordered by
// (score desc, best-chunk row asc).  Honours the row mask (label filter) and the score floor (nk_index_set_min_score: the
// reference keeps a node only if bestScore >= 0, call_vector.go:243).  Exact fp32 scores, no over-select loop: one pass
// with a per-node atomic max (segment-max), one top-k over the node keys.  Returns the number of nodes found (<= k).
int nk_search_groups(NkIndex *ix, const float *query_host, uint32_t k, uint32_t *out_group, uint32_t *out_row, float *out_score) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    if (k == 0 || s->n == 0) return 0;
    if (!query_host || !out_group || !out_row || !out_score) { nk::set_error("null argument"); return -1; }
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!s->group_on || ix->n_groups == 0) { nk::set_error("nk_search_groups: no row groups set (nk_index_set_row_groups)"); return -1; }
    const uint32_t G = ix->n_groups, ke = k < G ? k : G;
    if (ke > NK_MAX_K) { nk::set_error("nk_search_groups: k=%u exceeds NK_MAX_K=%u", ke, NK_MAX_K); return -1; }
    NK_CUDA_OK(cudaSetDevice(s->device));
    NK_RANGE_PUSH("nk_search_groups");
    struct Pop { ~Pop() { NK_RANGE_POP(); } } pop_on_exit;
    if (nk::ws_reserve((void **)&s->ws.queries, &s->ws.queries_bytes, (size_t)ix->dim * 4)) return -1;
    if (nk::ws_reserve(&s->ws.scratch, &s->ws.scratch_bytes, (size_t)G * 8)) return -1;
    if (nk::ws_reserve((void **)&s->ws.keys, &s->ws.keys_bytes, (size_t)ke * 8)) return -1;
    if (nk::ws_reserve((void **)&s->ws.out_idx, &s->ws.out_idx_bytes, (size_t)ke * 8)) return -1;
    if (nk::ws_reserve((void **)&s->ws.out_score, &s->ws.out_score_bytes, (size_t)ke * 4)) return -1;
    unsigned long long *best = static_cast<unsigned long long *>(s->ws.scratch);
    NK_CUDA_OK(cudaMemcpyAsync(s->ws.queries, query_host, (size_t)ix->dim * 4, cudaMemcpyHostToDevice, s->stream));
    NK_CUDA_OK(cudaMemsetAsync(best, 0, (size_t)G * 8, s->stream));
    if (nk::group_best(s->rows, ix->dtype, s->n, ix->dim, s->base, s->ws.queries, ix->metric, s->group, s->mask_on ? s->mask : nullptr,
                       ix->key_floor(), best, s->stream))
        return -1;
    if (nk::topk_keys(s->di, best, G, ke, s->ws, s->ws.keys, s->stream)) return -1;
    if (nk::decode_group_keys(s->ws.keys, ke, ix->metric, s->group, s->base, s->ws.out_idx, s->ws.out_idx + ke, s->ws.out_score, s->stream)) return -1;
    ix->stats.kernel_launches += 4;
    ix->stats.searches++; ix->stats.queries++;
    ix->stats.bytes_scanned += (uint64_t)s->n * ix->dim * ix->esz();
    NK_CUDA_OK(cudaMemcpyAsync(out_group, s->ws.out_idx, (size_t)ke * 4, cudaMemcpyDeviceToHost, s->stream));
    NK_CUDA_OK(cudaMemcpyAsync(out_row, s->ws.out_idx + ke, (size_t)ke * 4, cudaMemcpyDeviceToHost, s->stream));
    NK_CUDA_OK(cudaMemcpyAsync(out_score, s->ws.out_score, (size_t)ke * 4, cudaMemcpyDeviceToHost, s->stream));
    s->last_filter = false;
    if (finish_deferred(ix, *s) < 0) return -1;
    uint32_t found = 0;
    while (found < ke && out_group[found] != 0xffffffffu) ++found;
    return (int)found;
}

// ---- cluster-routed search (ClusterIndex.SearchWithClusters, kmeans.go:816-836; cluster_search.cu) ---------------------------
int nk_index_set_clusters(NkIndex *ix, const float *centroids_host, uint32_t K, const int32_t *assign_host, uint64_t n_rows) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    std::lock_guard<std::mutex> lk(ix->mu);
    if (!centroids_host) {
        s->clusters.on = false;
        return 0;
    }
    if (K == 0 || K > NK_MAX_CLUSTERS) { nk::set_error("nk_index_set_clusters: K=%u outside [1, NK_MAX_CLUSTERS=%u]", K, NK_MAX_CLUSTERS); return -1; }
    if (n_rows != s->n) { nk::set_error("nk_index_set_clusters: %llu assignments, index has %llu rows", (unsigned long long)n_rows, (unsigned long long)s->n); return -1; }
    if (n_rows && !assign_host) { nk::set_error("null argument"); return -1; }
    NK_CUDA_OK(cudaSetDevice(s->device));
    if (nk::cluster_layout_build(s->clusters, centroids_host, K, ix->dim, assign_host, n_rows, s->stream, &ix->stats.kernel_launches)) return -1;
    ix->stats.bytes_h2d += (uint64_t)K * ix->dim * 4 + n_rows * 4;
    return 0;
}

static int search_clusters_impl(NkIndex *ix, NkShard *s, const float *q_dev, uint32_t Q, uint32_t k, uint32_t n_probe, uint32_t *out_idx_dev,
                                float *out_score_dev, int32_t *out_probe_dev, cudaStream_t st) {
    nk::ClusterSearchArgs a;
    a.rows = s->rows; a.dtype = ix->dtype; a.dim = ix->dim; a.row_base = s->base;
    a.row_mask = s->mask_on ? s->mask : nullptr; a.min_score = ix->key_floor(); a.metric = ix->metric;
    a.queries = q_dev; a.Q = Q; a.k = k; a.n_probe = n_probe;
    a.out_idx = out_idx_dev; a.out_score = out_score_dev; a.out_probe = out_probe_dev;
    a.flags = s->ws.flags; a.stream = st;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;
    a.timing = ix->timing_on; a.timing_events = &ev;
    NK_RANGE_PUSH("nk_search_clusters");
    const int rc = nk::cluster_search(s->di, s->clusters, a, s->cws, &ix->stats.kernel_launches);
    NK_RANGE_POP();
    for (auto &e : ev) {
        s->timing.push_back(e);
        s->timing_launches.push_back(1);
    }
    ix->last_path = NK_PATH_SIMT;
    ix->stats.searches++;
    ix->stats.queries += Q;
    return rc;
}

// Shared argument checks; returns 1 when there is nothing to search (k == 0, Q == 0 or no rows), 0 to go on, -1 on error.
static int clusters_precheck(NkIndex *ix, NkShard *s, uint32_t Q, uint32_t k, uint32_t n_probe) {
    if (k > NK_MAX_K) { nk::set_error("nk_search_clusters: k=%u exceeds NK_MAX_K=%u", k, NK_MAX_K); return -1; }
    if (n_probe == 0) { nk::set_error("nk_search_clusters: n_probe must be >= 1"); return -1; }
    if (k == 0 || Q == 0 || s->n == 0) return 1;
    if (!s->clusters.on) { nk::set_error("nk_search_clusters: no clusters set (nk_index_set_clusters)"); return -1; }
    (void)ix;
    return 0;
}

int nk_search_clusters(NkIndex *ix, const float *queries_host, uint32_t Q, uint32_t k, uint32_t n_probe, uint32_t *out_idx, float *out_score,
                       int32_t *out_probe) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    std::lock_guard<std::mutex> lk(ix->mu);
    const int pre = clusters_precheck(ix, s, Q, k, n_probe);
    if (pre) return pre < 0 ? -1 : 0;
    if (!queries_host || !out_idx || !out_score) { nk::set_error("null argument"); return -1; }
    NK_CUDA_OK(cudaSetDevice(s->device));
    const uint32_t P = std::min(n_probe, s->clusters.K);
    const size_t qbytes = (size_t)Q * ix->dim * 4, rbytes = (size_t)Q * k * 4, pbytes = (size_t)Q * P * 4;
    if (nk::ws_reserve((void **)&s->ws.queries, &s->ws.queries_bytes, qbytes)) return -1;
    if (nk::ws_reserve((void **)&s->ws.out_idx, &s->ws.out_idx_bytes, rbytes + pbytes)) return -1;
    if (nk::ws_reserve((void **)&s->ws.out_score, &s->ws.out_score_bytes, rbytes)) return -1;
    int32_t *d_probe = reinterpret_cast<int32_t *>(s->ws.out_idx + (size_t)Q * k);
    const size_t need = 2 * rbytes + pbytes + sizeof(int) * nk::NK_FLAG_WORDS;
    if (s->h_res_bytes < need) {
        if (s->h_res) cudaFreeHost(s->h_res);
        s->h_res = nullptr; s->h_res_bytes = 0;
        NK_CUDA_OK(cudaMallocHost((void **)&s->h_res, need + need / 4));
        s->h_res_bytes = need + need / 4;
    }
    NK_CUDA_OK(cudaMemcpyAsync(s->ws.queries, queries_host, qbytes, cudaMemcpyHostToDevice, s->stream));
    ix->stats.bytes_h2d += qbytes;
    if (search_clusters_impl(ix, s, s->ws.queries, Q, k, n_probe, s->ws.out_idx, s->ws.out_score, d_probe, s->stream)) return -1;
    // results, probe lists and status words come back through one pinned buffer and ONE synchronisation
    int *hflags = reinterpret_cast<int *>(s->h_res + 2 * rbytes + pbytes);
    NK_CUDA_OK(cudaMemcpyAsync(s->h_res, s->ws.out_idx, rbytes + pbytes, cudaMemcpyDeviceToHost, s->stream));
    NK_CUDA_OK(cudaMemcpyAsync(s->h_res + rbytes + pbytes, s->ws.out_score, rbytes, cudaMemcpyDeviceToHost, s->stream));
    NK_CUDA_OK(cudaMemcpyAsync(hflags, s->ws.flags, sizeof(int) * nk::NK_FLAG_WORDS, cudaMemcpyDeviceToHost, s->stream));
    NK_CUDA_OK(cudaStreamSynchronize(s->stream));
    ix->stats.bytes_d2h += 2 * rbytes + pbytes;
    if (hflags[nk::FLAG_FATAL]) {
        cudaMemsetAsync(s->ws.flags, 0, sizeof(int), s->stream);
        nk::set_error("internal: candidate buffer overflow (flag=%d)", hflags[nk::FLAG_FATAL]);
        return -1;
    }
    memcpy(out_idx, s->h_res, rbytes);
    if (out_probe) memcpy(out_probe, s->h_res + rbytes, pbytes);
    memcpy(out_score, s->h_res + rbytes + pbytes, rbytes);
    return (int)std::min<uint64_t>(k, s->n);
}

int nk_search_clusters_device(NkIndex *ix, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t n_probe, uint32_t *out_idx_dev,
                              float *out_score_dev, int32_t *out_probe_dev, void *stream) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    std::lock_guard<std::mutex> lk(ix->mu);
    const int pre = clusters_precheck(ix, s, Q, k, n_probe);
    if (pre) return pre < 0 ? -1 : 0;
    if (!queries_dev || !out_idx_dev || !out_score_dev) { nk::set_error("null argument"); return -1; }
    NK_CUDA_OK(cudaSetDevice(s->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    if (search_clusters_impl(ix, s, queries_dev, Q, k, n_probe, out_idx_dev, out_score_dev, out_probe_dev, st)) return -1;
    return (int)std::min<uint64_t>(k, s->n);
}

// ---- row-sharded search with the exchange behind the ABI (exchange.cu) ----------------------------------------------------
// One rank per GPU (one process each, or several single-device indexes in one process): scan this rank's shard, push the
// Q*k candidate keys into every peer's buffer over NVLink, merge what the peers pushed.  Asynchronous on `stream`; every
// rank must make the same sequence of calls.  out_*_dev: [Q x k] on this rank's device, identical on every rank.
int nk_search_sharded_device(NkIndex *ix, NkComm *comm, const float *queries_dev, uint32_t Q, uint32_t k, uint32_t *out_idx_dev,
                             float *out_score_dev, void *stream) {
    nk::DeviceGuard _restore_device;
    NkShard *s;
    if (single_shard(ix, &s)) return -1;
    if (!comm) { nk::set_error("null communicator"); return -1; }
    if (k == 0 || Q == 0) return 0;
    cudaStream_t st = stream ? (cudaStream_t)stream : s->stream;
    {
        std::lock_guard<std::mutex> lk(ix->mu);
        NK_CUDA_OK(cudaSetDevice(s->device));
        if (nk::ws_reserve((void **)&s->ws.keys, &s->ws.keys_bytes, (size_t)Q * k * 8)) return -1;
    }
    if (nk_search_keys_device(ix, queries_dev, Q, k, s->ws.keys, st) < 0) return -1;
    if (nk_comm_exchange_merge(comm, s->ws.keys, Q, k, ix->metric, out_idx_dev, out_score_dev, st) < 0) return -1;
    ix->stats.kernel_launches += 2;
    return (int)k;
}

int nk_fill_uniform_device(int device_id, float *out_dev, uint64_t n_rows, uint32_t dim, uint64_t seed,
                           uint64_t row_base, void *stream) {
    nk::DeviceGuard _restore_device;
    NK_CUDA_OK(cudaSetDevice(device_id));
    return nk::fill_uniform(out_dev, NK_DTYPE_F32, n_rows, dim, seed, row_base, (cudaStream_t)stream);
}

}  // extern "C"
