// merge.cu — candidate-list merge, key decoding, and device top-k over a precomputed score array.
//
// merge_keys is the "partial top-k merge" step of the path: per-CTA lists inside one GPU, and the
// per-GPU lists of a row-sharded corpus (SURVEY.md §8e).  It applies the same (score desc, row asc)
// order as the scan, so the result does not depend on how rows were partitioned.
// topk_scores replaces the host insertion sort of cuda_topk (pkg/gpu/cuda/cuda_bridge.go:327-375):
// selection happens on the device and only k (index, score) pairs cross PCIe instead of n scores.
#include "kernels.cuh"

namespace nk {

constexpr int MERGE_THREADS = 256;
constexpr int MERGE_P = 2048;  // sort width; NK_MAX_K <= MERGE_P / 2

struct MergeParams {
    const uint64_t *keys;
    uint32_t n_lists;
    size_t list_stride, q_stride;
    uint32_t k;
    uint64_t *out;  // [Q][k]
    const int *only_if;
    uint32_t list_len;  // entries per input list (may differ from the output k)
    uint32_t *dec_idx;  // optional fused decode
    float *dec_score;
    int dec_metric;
    // optional: the lists are being written by PEER GPUs (exchange.cu); list l is complete once wait_flags[l] >= wait_epoch
    const uint32_t *wait_flags;
    uint32_t wait_epoch;
    int *wait_err;  // set to 2 if a peer did not arrive within ~2 s (never spin forever: a hung GPU is a strike)
    const uint32_t *q_lists;  // optional: query q merges only its first q_lists[q] lists (cluster-routed search)
};

// One CTA per query.  Streams the n_lists*k candidate keys through a 2048-wide sort buffer, keeping
// the best k at the front after every round.  Keys below the current k-th best are dropped on load.
__global__ void __launch_bounds__(MERGE_THREADS) merge_keys_kernel(MergeParams p) {
    pdl_trigger();
    pdl_wait();  // programmatic dependent of the scan / push kernel before it (common.cuh)
    if (p.only_if && *p.only_if == 0) return;
    __shared__ uint64_t sbuf[2 * MERGE_P];  // sort buffer (MERGE_P wide); the pre-filter caches up to 2 * MERGE_P whole keys here
    __shared__ int s_fill;
    const uint32_t q = blockIdx.x;
    const uint64_t *base = p.keys + (size_t)q * p.q_stride;
    const uint64_t total = (uint64_t)(p.q_lists ? p.q_lists[q] : p.n_lists) * p.list_len;
    const int tid = threadIdx.x;
    if (p.wait_flags) {
        // fused exchange wait: thread l polls peer l's arrival word (system-scope acquire), bounded by a wall-clock timeout
        if (tid < (int)p.n_lists) {
            unsigned long long t0, t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
            for (;;) {
                uint32_t v;
                asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p.wait_flags + tid) : "memory");
                if ((int32_t)(v - p.wait_epoch) >= 0) break;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > 2000000000ull) {
                    atomicExch(p.wait_err, 2);
                    break;
                }
                __nanosleep(64);
            }
        }
        __syncthreads();
    }

    // ---- pre-filter (many more keys than k, e.g. the 391 per-CTA lists of a small-shard CUDA-core scan): radix-select the
    // k-th largest SCORE WORD over all keys first (score words cached in shared memory, 8 bits per pass), so that only the k
    // best (+ ties) go through the sort — a 2048-wide bitonic network for k = 10 was most of a configs[0] search.
    uint64_t kth = 0;  // current k-th best key (0 = none yet): keys <= kth are dropped on load
    __shared__ int m_hist[256];
    __shared__ uint32_t m_prefix, m_red[2][MERGE_THREADS / 32];
    __shared__ int m_krem;
    if (total >= 4ull * p.k && total > 512 && total <= 2ull * MERGE_P) {
        const int n = (int)total, lane = tid & 31, warp = tid >> 5;
        uint32_t umax = 0u, umin = 0xffffffffu;
        for (int i0 = tid; i0 < n; i0 += 4 * MERGE_THREADS) {
            uint64_t h[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * MERGE_THREADS;
                const uint32_t l = (uint32_t)(i / (int)p.list_len), sl = (uint32_t)(i - (int)(l * p.list_len));
                h[u] = i < n ? __ldcg(base + (size_t)l * p.list_stride + sl) : 0ull;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * MERGE_THREADS;
                if (i < n) { sbuf[i] = h[u]; umax = max(umax, (uint32_t)(h[u] >> 32)); if (h[u]) umin = min(umin, (uint32_t)(h[u] >> 32)); }  // (empty slots stay out of the digit range: fewer passes)
            }
        }
        umax = __reduce_max_sync(0xffffffffu, umax);
        umin = __reduce_min_sync(0xffffffffu, umin);
        if (lane == 0) { m_red[0][warp] = umax; m_red[1][warp] = umin; }
        if (tid == 0) m_krem = (int)p.k;
        __syncthreads();
#pragma unroll
        for (int w = 0; w < MERGE_THREADS / 32; ++w) { umax = max(umax, m_red[0][w]); umin = min(umin, m_red[1][w]); }
        int rem = 32 - __clz(umax ^ umin);
        if (tid == 0) m_prefix = rem >= 32 ? 0u : (umax >> rem) << rem;
        __syncthreads();
        while (rem > 10) {  // (<= 10 unresolved low bits: the prefix is a lower bound of the k-th score word — a few more keys reach the sort)
            const int w = rem < 8 ? rem : 8, shift = rem - w;
            m_hist[tid] = 0;  // MERGE_THREADS == 256
            __syncthreads();
            const uint32_t prefix = m_prefix;
            for (int i = tid; i < n; i += MERGE_THREADS) {
                const uint32_t hi = (uint32_t)(sbuf[i] >> 32);
                if (rem >= 32 || (hi >> rem) == (prefix >> rem)) atomicAdd(&m_hist[(hi >> shift) & ((1u << w) - 1u)], 1);
            }
            __syncthreads();
            if (warp == 0) {  // digit holding the krem-th largest: lane l owns the 8 digits below nb - 8l, descending
                const int krem = m_krem, nb = 1 << w;
                int loc[8], sum = 0;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int dgt = nb - 1 - (lane * 8 + j);
                    loc[j] = dgt >= 0 ? m_hist[dgt] : 0;
                    sum += loc[j];
                }
                __syncwarp();
                int incl = sum;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                int c = incl - sum;
                if (c < krem && incl >= krem) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        if (c + loc[j] >= krem) {
                            m_prefix = prefix | ((uint32_t)(nb - 1 - (lane * 8 + j)) << shift);
                            m_krem = krem - c;
                            break;
                        }
                        c += loc[j];
                    }
                }
            }
            __syncthreads();
            rem = shift;
        }
        const uint32_t kth_hi = m_prefix;  // the k-th largest score word: keys with a smaller one cannot be in the top k
        if (kth_hi) kth = ((uint64_t)kth_hi << 32) - 1ull;
        // compact the survivors to the front of the buffer IN PLACE (every thread holds its keys in registers across the
        // barrier), sort just those, write the result: no second pass over the lists
        uint64_t mine[2 * MERGE_P / MERGE_THREADS];
#pragma unroll
        for (int u = 0; u < 2 * MERGE_P / MERGE_THREADS; ++u) {
            const int i = tid + u * MERGE_THREADS;
            mine[u] = i < n ? sbuf[i] : 0ull;
        }
        if (tid == 0) s_fill = 0;
        __syncthreads();
#pragma unroll
        for (int u = 0; u < 2 * MERGE_P / MERGE_THREADS; ++u)
            if (mine[u] > kth) {
                const int slot = atomicAdd(&s_fill, 1);
                if (slot < MERGE_P) sbuf[slot] = mine[u];
            }
        __syncthreads();
        if (s_fill <= MERGE_P) {  // (more than MERGE_P keys tie on the k-th score word: take the general path below)
            const int filled = s_fill;
            int Ps = 32;
            while (Ps < filled) Ps <<= 1;
            for (int i = filled + tid; i < Ps; i += MERGE_THREADS) sbuf[i] = 0ull;
            block_bitonic_sort_desc(sbuf, Ps);
            for (uint32_t i = tid; i < p.k; i += MERGE_THREADS) {
                const uint64_t key = (int)i < filled ? sbuf[i] : 0ull;
                if (p.out) p.out[(size_t)q * p.k + i] = key;
                if (p.dec_idx) {
                    float sc = key_score(key);
                    if (p.dec_metric == NK_METRIC_EUCLIDEAN) sc = sqrtf(fmaxf(-sc, 0.0f));
                    p.dec_idx[(size_t)q * p.k + i] = key ? key_row(key) : 0xffffffffu;
                    p.dec_score[(size_t)q * p.k + i] = key ? sc : 0.0f;
                }
            }
            return;
        }
        __syncthreads();
    }

    // sort width: the whole input when it fits a smaller power of two (cross-GPU merges fold a few dozen keys)
    int P = MERGE_P;
    if (total <= (uint64_t)MERGE_P) {
        P = 64;
        while ((uint64_t)P < total || P < (int)p.k) P <<= 1;
    }
    for (int i = tid; i < P; i += MERGE_THREADS) sbuf[i] = 0ull;
    if (tid == 0) s_fill = 0;
    __syncthreads();

    uint64_t pos = 0;
    while (pos < total) {
        // fill slots [fill, MERGE_P) with keys that can still matter
        const uint64_t room_all = (uint64_t)P - (uint64_t)s_fill;
        __syncthreads();
        const int fill0 = s_fill;
        uint64_t chunk = total - pos;
        if (chunk > room_all) chunk = room_all;
        for (uint64_t i = tid; i < chunk; i += MERGE_THREADS) {
            uint64_t g = pos + i;
            uint32_t l = (uint32_t)(g / p.list_len), s = (uint32_t)(g - (uint64_t)l * p.list_len);
            uint64_t key = __ldcg(base + (size_t)l * p.list_stride + s);  // L2: peer GPUs may have just written it
            if (key > kth) {
                int slot = atomicAdd(&s_fill, 1);
                sbuf[slot] = key;
            }
        }
        pos += chunk;
        __syncthreads();
        const int filled = s_fill;
        // sort only when the buffer is nearly full or the input is exhausted
        if (pos >= total || filled > P - MERGE_THREADS) {
            int Ps = 32;  // sort only as wide as the live keys (a pre-filtered input leaves k + ties of them)
            while (Ps < filled) Ps <<= 1;
            if (Ps > P) Ps = P;
            for (int i = filled + tid; i < Ps; i += MERGE_THREADS) sbuf[i] = 0ull;
            block_bitonic_sort_desc(sbuf, Ps);
            int keep = filled < (int)p.k ? filled : (int)p.k;
            if (filled >= (int)p.k) kth = sbuf[p.k - 1];
            __syncthreads();
            if (tid == 0) s_fill = keep;
            __syncthreads();
        }
        (void)fill0;
    }
    __syncthreads();
    const int have = s_fill;
    for (uint32_t i = tid; i < p.k; i += MERGE_THREADS) {
        const uint64_t key = (int)i < have ? sbuf[i] : 0ull;
        if (p.out) p.out[(size_t)q * p.k + i] = key;
        if (p.dec_idx) {
            float sc = key_score(key);
            if (p.dec_metric == NK_METRIC_EUCLIDEAN) sc = sqrtf(fmaxf(-sc, 0.0f));
            p.dec_idx[(size_t)q * p.k + i] = key ? key_row(key) : 0xffffffffu;
            p.dec_score[(size_t)q * p.k + i] = key ? sc : 0.0f;
        }
    }
}

int merge_keys(const uint64_t *keys, uint32_t n_lists, size_t list_stride, size_t q_stride, uint32_t Q, uint32_t k,
               uint64_t *out_keys, cudaStream_t stream, const int *only_if, uint32_t list_len, uint32_t *dec_idx, float *dec_score,
               int dec_metric, const uint32_t *wait_flags, uint32_t wait_epoch, int *wait_err, const uint32_t *q_lists) {
    if (Q == 0 || k == 0) return 0;
    if (k > MERGE_P / 2) {
        set_error("merge: k=%u too large", k);
        return -1;
    }
    if (wait_flags && n_lists > MERGE_THREADS) {
        set_error("merge: too many peers");
        return -1;
    }
    MergeParams p{keys, n_lists, list_stride, q_stride, k, out_keys, only_if, list_len ? list_len : k, dec_idx, dec_score, dec_metric,
                  wait_flags, wait_epoch, wait_err, q_lists};
    NK_CUDA_OK(launch_pdl(merge_keys_kernel, dim3(Q), dim3(MERGE_THREADS), 0, stream, true, p));
    return 0;
}

__global__ void decode_keys_kernel(const uint64_t *keys, size_t total, int metric, uint32_t *out_idx, float *out_score,
                                   const int *only_if) {
    if (only_if && *only_if == 0) return;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    uint64_t key = keys[i];
    float s = key_score(key);
    if (metric == NK_METRIC_EUCLIDEAN) s = sqrtf(fmaxf(-s, 0.0f));
    out_idx[i] = key ? key_row(key) : 0xffffffffu;
    out_score[i] = key ? s : 0.0f;
}

int decode_keys(const uint64_t *keys, uint32_t Q, uint32_t k, int metric, uint32_t *out_idx, float *out_score,
                cudaStream_t stream, const int *only_if) {
    size_t total = (size_t)Q * k;
    if (total == 0) return 0;
    decode_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(keys, total, metric, out_idx, out_score, only_if);
    NK_CUDA_OK(cudaGetLastError());
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Device top-k over a score array (legacy cuda_topk).  Same threshold + buffer + prune scheme as the
// fused scan, fed from memory instead of from the dot products.
// ---------------------------------------------------------------------------------------------
constexpr int TOPK_THREADS = 256;
constexpr int TOPK_IV = 1024;  // scores per CTA between prune checks

__global__ void __launch_bounds__(TOPK_THREADS) topk_scores_kernel(const float *scores, uint32_t n, uint32_t k, int P,
                                                                   uint64_t *cand, uint64_t *partial, int *flags,
                                                                   const uint64_t *below) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(smem_raw);
    __shared__ float s_tau;
    __shared__ int s_cnt;
    if (threadIdx.x == 0) {
        s_tau = -INFINITY;
        s_cnt = 0;
    }
    __syncthreads();
    uint64_t *my = cand + (size_t)blockIdx.x * P;
    const uint32_t num_iv = (n + TOPK_IV - 1) / TOPK_IV;
    for (uint32_t iv = blockIdx.x; iv < num_iv; iv += gridDim.x) {
        for (uint32_t i = iv * TOPK_IV + threadIdx.x; i < (iv + 1) * TOPK_IV && i < n; i += TOPK_THREADS) {
            float s = scores[i];
            if (s != s) s = -INFINITY;
            if (s >= s_tau) {
                const uint64_t key = make_key(s, i);
                if (!below || key < below[0]) {
                    int pos = atomicAdd(&s_cnt, 1);
                    if (pos < P) my[pos] = key;
                    else atomicExch(flags, 1);
                }
            }
        }
        __syncthreads();
        bool need = s_cnt > P - TOPK_IV;
        __syncthreads();
        if (need) block_prune(my, P, &s_cnt, &s_tau, k, sbuf, P);
    }
    block_prune(my, P, &s_cnt, &s_tau, k, sbuf, P);
    for (uint32_t i = threadIdx.x; i < k; i += TOPK_THREADS) partial[(size_t)blockIdx.x * k + i] = sbuf[i];
}

// Top-k over an array of ready-made keys (0 = empty): the node-level selection of the best-of-chunks search
// (group_best fills one key per node).  Same threshold + buffer + prune scheme as topk_scores_kernel.
__global__ void __launch_bounds__(TOPK_THREADS) topk_keys_kernel(const unsigned long long *keys, uint32_t n, uint32_t k, int P,
                                                                 uint64_t *cand, uint64_t *partial, int *flags) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(smem_raw);
    __shared__ float s_tau;
    __shared__ int s_cnt;
    if (threadIdx.x == 0) {
        s_tau = -INFINITY;
        s_cnt = 0;
    }
    __syncthreads();
    uint64_t *my = cand + (size_t)blockIdx.x * P;
    const uint32_t num_iv = (n + TOPK_IV - 1) / TOPK_IV;
    for (uint32_t iv = blockIdx.x; iv < num_iv; iv += gridDim.x) {
        for (uint32_t i = iv * TOPK_IV + threadIdx.x; i < (iv + 1) * TOPK_IV && i < n; i += TOPK_THREADS) {
            const uint64_t key = keys[i];
            if (key && key_score(key) >= s_tau) {
                int pos = atomicAdd(&s_cnt, 1);
                if (pos < P) my[pos] = key;
                else atomicExch(flags, 1);
            }
        }
        __syncthreads();
        bool need = s_cnt > P - TOPK_IV;
        __syncthreads();
        if (need) block_prune(my, P, &s_cnt, &s_tau, k, sbuf, P);
    }
    block_prune(my, P, &s_cnt, &s_tau, k, sbuf, P);
    for (uint32_t i = threadIdx.x; i < k; i += TOPK_THREADS) partial[(size_t)blockIdx.x * k + i] = sbuf[i];
}
// keys [k] -> (group, row, score): group = group_of_row[row - row_base]
__global__ void decode_group_keys_kernel(const uint64_t *keys, uint32_t k, int metric, const uint32_t *group, uint64_t row_base,
                                         uint32_t *out_group, uint32_t *out_row, float *out_score) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= k) return;
    const uint64_t key = keys[i];
    float s = key_score(key);
    if (metric == NK_METRIC_EUCLIDEAN) s = sqrtf(fmaxf(-s, 0.0f));
    const uint32_t row = key_row(key);
    out_group[i] = key ? group[row - (uint32_t)row_base] : 0xffffffffu;
    out_row[i] = key ? row : 0xffffffffu;
    out_score[i] = key ? s : 0.0f;
}

__global__ void update_below_kernel(const uint64_t *keys, uint32_t Q, uint32_t k, uint64_t *below) {
    uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q < Q) below[q] = keys[(size_t)q * k + k - 1];  // 0 when the pass ran dry: nothing is below key 0
}
int update_below(const uint64_t *keys, uint32_t Q, uint32_t k, uint64_t *below, cudaStream_t s) {
    update_below_kernel<<<(Q + 127) / 128, 128, 0, s>>>(keys, Q, k, below);
    NK_CUDA_OK(cudaGetLastError());
    return 0;
}

int topk_keys(const DeviceInfo &di, const unsigned long long *keys, uint32_t n, uint32_t k, Workspace &ws, uint64_t *out_keys,
              cudaStream_t s) {
    if (n == 0 || k == 0) return 0;
    if (k > NK_MAX_K) {
        set_error("k=%u exceeds NK_MAX_K=%u", k, NK_MAX_K);
        return -1;
    }
    int P = (int)next_pow2(k + TOPK_IV + 1);
    uint32_t num_iv = (n + TOPK_IV - 1) / TOPK_IV;
    uint32_t grid = (uint32_t)di.num_sms * 2;
    if (grid > num_iv) grid = num_iv;
    if (ws_reserve((void **)&ws.cand, &ws.cand_bytes, (size_t)grid * P * 8)) return -1;
    if (ws_reserve((void **)&ws.partial, &ws.partial_bytes, (size_t)grid * k * 8)) return -1;
    size_t smem = (size_t)P * 8;
    NK_CUDA_OK(cudaFuncSetAttribute(topk_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topk_keys_kernel<<<grid, TOPK_THREADS, smem, s>>>(keys, n, k, P, ws.cand, ws.partial, ws.flags);
    NK_CUDA_OK(cudaGetLastError());
    return merge_keys(ws.partial, grid, k, 0, 1, k, out_keys, s);
}
int decode_group_keys(const uint64_t *keys, uint32_t k, int metric, const uint32_t *group, uint64_t row_base, uint32_t *out_group,
                      uint32_t *out_row, float *out_score, cudaStream_t s) {
    if (k == 0) return 0;
    decode_group_keys_kernel<<<(k + 127) / 128, 128, 0, s>>>(keys, k, metric, group, row_base, out_group, out_row, out_score);
    NK_CUDA_OK(cudaGetLastError());
    return 0;
}

int topk_scores(const DeviceInfo &di, const float *scores, uint32_t n, uint32_t k, Workspace &ws, uint64_t *out_keys,
                cudaStream_t s, const uint64_t *below) {
    if (n == 0 || k == 0) return 0;
    if (k > NK_MAX_K) {
        set_error("k=%u exceeds NK_MAX_K=%u", k, NK_MAX_K);
        return -1;
    }
    int P = (int)next_pow2(k + TOPK_IV + 1);
    uint32_t num_iv = (n + TOPK_IV - 1) / TOPK_IV;
    uint32_t grid = (uint32_t)di.num_sms * 2;
    if (grid > num_iv) grid = num_iv;
    if (ws_reserve((void **)&ws.cand, &ws.cand_bytes, (size_t)grid * P * 8)) return -1;
    if (ws_reserve((void **)&ws.partial, &ws.partial_bytes, (size_t)grid * k * 8)) return -1;
    size_t smem = (size_t)P * 8;
    NK_CUDA_OK(cudaFuncSetAttribute(topk_scores_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    topk_scores_kernel<<<grid, TOPK_THREADS, smem, s>>>(scores, n, k, P, ws.cand, ws.partial, ws.flags, below);
    NK_CUDA_OK(cudaGetLastError());
    return merge_keys(ws.partial, grid, k, 0, 1, k, out_keys, s);
}

}  // namespace nk
