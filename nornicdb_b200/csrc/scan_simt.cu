// scan_simt.cu — fused distance + top-k scan on CUDA cores (the HBM-bound small-Q path).
//
// Replaces, in one kernel, the reference's per-query chain
//   cublasSgemv (cuda_bridge.go:302-309) -> D2H of all n scores -> host insertion top-k (cuda_bridge.go:336-371)
// and the CPU scan simd.Batch{Cosine,Dot,Euclidean} + bounded top-k (pkg/simd/simd.go:149-231).
//
// Shape of the work: every corpus byte is read from HBM exactly once per group of QT<=8 queries.
//   * a warp owns R rows at a time; lanes stride the row in 16-byte vectors (float4 / 8 halves), so a
//     warp-wide load is one fully coalesced 512 B segment per row;
//   * the QT queries of the group live in shared memory (read as conflict-free LDS.128, re-used by the
//     R rows in registers);
//   * R*QT partial dot products per lane are folded with a butterfly "reduce-scatter" (31 shuffles for
//     32 values) so each lane ends up owning one finished (row, query) score;
//   * scores never go to memory: the owner lane compares against the query's running threshold (k-th
//     best score this CTA has seen) and only then appends a packed 64-bit key to a per-(CTA, query)
//     candidate buffer; the CTA prunes a buffer with a bitonic sort when it could overflow;
//   * each CTA finally emits its best k keys per query; merge_keys() folds the per-CTA lists.
//
// Algorithmic HBM traffic per launch = n*dim*sizeof(elem) (+ QT*dim*4 of queries): DESIGN.md §Kernels.
#include <map>
#include <mutex>
#include <tuple>

#include "simt_lane.cuh"

namespace nk {

constexpr int SIMT_THREADS = 256;
constexpr int SIMT_WARPS = SIMT_THREADS / 32;
constexpr int SIMT_RT = 256;  // rows a CTA scores between two prune checks

struct SimtParams {
    const void *rows;
    uint32_t n, dim;
    uint64_t row_base;
    const float *queries;  // [Q x dim], this launch handles queries q0 .. q0+nq-1
    uint32_t q0, nq, k;
    int metric;
    int P;               // candidate-buffer capacity = sort width (power of two)
    uint64_t *cand;      // [grid][QT][P]
    uint64_t *partial;   // [Q][grid][k]
    int *flags;
    const int *only_if;  // device-side conditional fallback: run only if *only_if != 0
    const uint64_t *below;  // per-query exclusive key bound (k > NK_MAX_K passes) or nullptr
    const uint32_t *mask;   // row bitmask or nullptr
    float min_score;        // caller's score floor (key space); -inf = none
};

template <typename T, bool VEC, int QT, int R, bool EUCLID>
__global__ void __launch_bounds__(SIMT_THREADS) knn_scan_simt_kernel(SimtParams p) {
    pdl_trigger();  // the merge launch behind this scan may begin (it waits for this grid before reading)
    pdl_wait();     // exact-stage twin of a filter search: programmatic dependent of the finish kernel
    if (p.only_if && *p.only_if == 0) return;
    using L = Lane<T, VEC>;
    constexpr int EPL = L::EPL;
    constexpr int CH = 32 * EPL;  // elements a warp covers per step
    constexpr int V = R * QT;
    static_assert(V <= 32 && (32 % V) == 0, "R*QT must divide 32");
    constexpr int LPV = 32 / V;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(smem_raw);
    float *qs = reinterpret_cast<float *>(smem_raw + (size_t)p.P * 8);  // [QT][dim]
    __shared__ float s_qq[QT];
    __shared__ float s_tau[QT];
    __shared__ int s_cnt[QT];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t dim = p.dim, n = p.n;
    const T *rows = static_cast<const T *>(p.rows);

    // ---- stage the query group -----------------------------------------------------------------
    for (uint32_t i = tid; i < (uint32_t)QT * dim; i += SIMT_THREADS) {
        uint32_t qi = i / dim, j = i - qi * dim;
        qs[i] = qi < p.nq ? p.queries[(size_t)(p.q0 + qi) * dim + j] : 0.0f;
    }
    if (tid < QT) {
        s_tau[tid] = p.min_score;
        s_cnt[tid] = 0;
    }
    __syncthreads();
    for (int qi = warp; qi < QT; qi += SIMT_WARPS) {  // |q|^2 per query (cosine)
        float a = 0.0f;
        for (uint32_t j = lane; j < dim; j += 32) a = fmaf(qs[qi * dim + j], qs[qi * dim + j], a);
#pragma unroll
        for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) s_qq[qi] = a;
    }
    __syncthreads();

    uint64_t *my_cand = p.cand + (size_t)blockIdx.x * QT * p.P;
    const int prune_at = p.P - SIMT_RT;
    const uint32_t num_iv = (n + SIMT_RT - 1) / SIMT_RT;
    const uint32_t nsteps = (dim + CH - 1) / CH;

    for (uint32_t iv = blockIdx.x; iv < num_iv; iv += gridDim.x) {
        const uint32_t base = iv * SIMT_RT;
#pragma unroll 1
        for (int t = 0; t < SIMT_RT / (SIMT_WARPS * R); ++t) {
            const uint32_t row0 = base + (uint32_t)(t * SIMT_WARPS + warp) * R;
            if (row0 >= n) continue;  // warp-uniform
            const T *rp[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                uint32_t rr = row0 + r < n ? row0 + r : n - 1;  // clamp; masked below
                rp[r] = rows + (size_t)rr * dim;
            }
            float acc[V];
            float xx[R];
#pragma unroll
            for (int i = 0; i < V; ++i) acc[i] = 0.0f;
#pragma unroll
            for (int r = 0; r < R; ++r) xx[r] = 0.0f;

#pragma unroll 2
            for (uint32_t c = 0; c < nsteps; ++c) {
                const uint32_t e = c * CH + lane * EPL;
                if (e < dim) {
                    float x[R][EPL];
#pragma unroll
                    for (int r = 0; r < R; ++r) L::load(rp[r] + e, x[r]);
#pragma unroll
                    for (int qi = 0; qi < QT; ++qi) {
                        float q[EPL];
                        if constexpr (EPL == 1) {
                            q[0] = qs[qi * dim + e];
                        } else {
#pragma unroll
                            for (int h = 0; h < EPL / 4; ++h) {
                                float4 t4 = *reinterpret_cast<const float4 *>(&qs[qi * dim + e + 4 * h]);
                                q[4 * h + 0] = t4.x; q[4 * h + 1] = t4.y; q[4 * h + 2] = t4.z; q[4 * h + 3] = t4.w;
                            }
                        }
#pragma unroll
                        for (int r = 0; r < R; ++r) {
#pragma unroll
                            for (int u = 0; u < EPL; ++u) {
                                if constexpr (EUCLID) {
                                    float d = x[r][u] - q[u];
                                    acc[r * QT + qi] = fmaf(d, d, acc[r * QT + qi]);
                                } else {
                                    acc[r * QT + qi] = fmaf(x[r][u], q[u], acc[r * QT + qi]);
                                }
                            }
                        }
                    }
                    if constexpr (!EUCLID) {
#pragma unroll
                        for (int r = 0; r < R; ++r)
#pragma unroll
                            for (int u = 0; u < EPL; ++u) xx[r] = fmaf(x[r][u], x[r][u], xx[r]);
                    }
                }
            }

            // ---- fold across lanes; lane owns (row r, query qi) -----------------------------------
            warp_reduce_scatter<V>(acc, lane);
            const int j = lane / LPV;
            const int r = j / QT, qi = j - r * QT;
            float s = acc[0];
            float xr = 0.0f;
            if constexpr (!EUCLID) {
                warp_reduce_scatter<R>(xx, lane);
                xr = __shfl_sync(0xffffffffu, xx[0], r * (32 / R));
            }
            const uint32_t row = row0 + r;
            if ((lane % LPV) == 0 && row < n && (uint32_t)qi < p.nq && (!p.mask || ((p.mask[row >> 5] >> (row & 31)) & 1u))) {
                if constexpr (EUCLID) {
                    s = -s;
                } else if (p.metric == NK_METRIC_COSINE) {
                    // dot / sqrt(|x|^2 |q|^2); zero vector -> 0 (simd_amd64.go:31-35 NaN -> 0)
                    float den = sqrtf(xr * s_qq[qi]);
                    s = den > 0.0f ? s / den : 0.0f;
                }
                if (s != s) s = -INFINITY;
                if (s >= s_tau[qi] && s >= p.min_score) {  // (a prune with fewer than k live keys resets tau to -inf)
                    const uint64_t key = make_key(s, (uint32_t)(p.row_base + row));
                    if (!p.below || key < p.below[p.q0 + qi]) {
                        int pos = atomicAdd(&s_cnt[qi], 1);
                        if (pos < p.P) my_cand[(size_t)qi * p.P + pos] = key;
                        else atomicExch(p.flags, 1);
                    }
                }
            }
        }
        // ---- prune any buffer that could overflow during the next interval ---------------------
        __syncthreads();
        uint32_t need = 0;
#pragma unroll
        for (int qi = 0; qi < QT; ++qi) need |= (s_cnt[qi] > prune_at ? 1u : 0u) << qi;
        __syncthreads();
        if (need && p.P == 512) {
            // k <= 255: warp w prunes query w with the register radix select (QT <= 8 queries, 8 warps: all in parallel, ~2 us)
            if (warp < QT && (need & (1u << warp)))
                warp_prune<16>(my_cand + (size_t)warp * p.P, &s_cnt[warp], &s_tau[warp], p.k, lane, nullptr, 0, false, 0.0f, (int)p.k, p.min_score);
            __syncthreads();
        } else if (need) {
#pragma unroll 1
            for (int qi = 0; qi < QT; ++qi)
                if (need & (1u << qi)) block_prune(my_cand + (size_t)qi * p.P, p.P, &s_cnt[qi], &s_tau[qi], p.k, sbuf, p.P);
        }
    }

    // ---- emit this CTA's best k per query --------------------------------------------------------
    if (p.P == 512) {
        // k <= 255: one warp per query selects the best k of the (<= 512) buffered keys with the register radix select
        // (~2 us) instead of a 45-stage block bitonic sort — on small shards (configs[0]: one interval per CTA) the
        // emission sort WAS the scan time.  The list goes out unsorted; merge_keys sorts.
        __syncthreads();
        for (uint32_t qi = warp; qi < p.nq; qi += SIMT_WARPS) {
            uint64_t *dst = p.partial + ((size_t)(p.q0 + qi) * gridDim.x + blockIdx.x) * p.k;
            warp_prune<16>(my_cand + (size_t)qi * p.P, &s_cnt[qi], &s_tau[qi], p.k, lane, dst, (int)p.k, false, 0.0f, (int)p.k, p.min_score);
        }
        return;
    }
#pragma unroll 1
    for (uint32_t qi = 0; qi < p.nq; ++qi) {
        block_prune(my_cand + (size_t)qi * p.P, p.P, &s_cnt[qi], &s_tau[qi], p.k, sbuf, p.P);
        uint64_t *dst = p.partial + ((size_t)(p.q0 + qi) * gridDim.x + blockIdx.x) * p.k;
        for (uint32_t i = tid; i < p.k; i += SIMT_THREADS) dst[i] = sbuf[i];  // zeros beyond the live entries
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
typedef void (*SimtKernel)(SimtParams);

template <typename T, bool VEC, bool EUCLID>
static SimtKernel pick_qt(int qt) {
    if constexpr (VEC) {
        switch (qt) {
            case 8: return knn_scan_simt_kernel<T, VEC, 8, 4, EUCLID>;
            case 4: return knn_scan_simt_kernel<T, VEC, 4, 8, EUCLID>;
            case 2: return knn_scan_simt_kernel<T, VEC, 2, 8, EUCLID>;
            default: return knn_scan_simt_kernel<T, VEC, 1, 8, EUCLID>;
        }
    } else {
        switch (qt) {
            case 4: return knn_scan_simt_kernel<T, VEC, 4, 8, EUCLID>;
            default: return knn_scan_simt_kernel<T, VEC, 1, 8, EUCLID>;
        }
    }
}

static SimtKernel pick_kernel(int dtype, bool vec, bool euclid, int qt) {
    if (dtype == NK_DTYPE_F16) {
        if (vec) return euclid ? pick_qt<__half, true, true>(qt) : pick_qt<__half, true, false>(qt);
        return euclid ? pick_qt<__half, false, true>(qt) : pick_qt<__half, false, false>(qt);
    }
    if (dtype == NK_DTYPE_BF16) {
        if (vec) return euclid ? pick_qt<__nv_bfloat16, true, true>(qt) : pick_qt<__nv_bfloat16, true, false>(qt);
        return euclid ? pick_qt<__nv_bfloat16, false, true>(qt) : pick_qt<__nv_bfloat16, false, false>(qt);
    }
    if (vec) return euclid ? pick_qt<float, true, true>(qt) : pick_qt<float, true, false>(qt);
    return euclid ? pick_qt<float, false, true>(qt) : pick_qt<float, false, false>(qt);
}

// cudaFuncSetAttribute + occupancy query once per (kernel, device, smem) instead of once per search
static std::mutex g_simt_mu;
static std::map<std::tuple<const void *, int, size_t>, int> g_simt_occ;
static std::map<std::pair<const void *, int>, size_t> g_simt_smem;
static int simt_ensure(const void *kern, int device, size_t smem) {
    std::lock_guard<std::mutex> lk(g_simt_mu);
    size_t &cur = g_simt_smem[{kern, device}];
    if (cur < smem || cur == 0) {
        NK_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cur = smem;
    }
    return 0;
}
static int simt_occupancy(const void *kern, int device, size_t smem) {
    std::lock_guard<std::mutex> lk(g_simt_mu);
    auto key = std::make_tuple(kern, device, smem);
    auto it = g_simt_occ.find(key);
    if (it != g_simt_occ.end()) return it->second;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SIMT_THREADS, smem) != cudaSuccess) { cudaGetLastError(); occ = 1; }
    if (occ < 1) occ = 1;
    if (occ > 8) occ = 8;
    g_simt_occ[key] = occ;
    return occ;
}

int simt_cap_for_k(uint32_t k) {
    uint32_t P = next_pow2(k + SIMT_RT + 1);
    return (int)(P < 512 ? 512 : P);
}

int scan_simt(const DeviceInfo &di, const ScanArgs &a, Workspace &ws, uint64_t *out_keys, uint64_t *launches) {
    if (a.n == 0 || a.Q == 0 || a.k == 0) return 0;
    if (a.k > NK_MAX_K) {
        set_error("k=%u exceeds NK_MAX_K=%u", a.k, NK_MAX_K);
        return -1;
    }
    const size_t esz = a.dtype == NK_DTYPE_F32 ? 4 : 2;
    const uint32_t vec_elems = a.dtype == NK_DTYPE_F32 ? 4 : 8;
    const bool vec = (a.dim % vec_elems == 0) && ((reinterpret_cast<uintptr_t>(a.rows) & 15) == 0);
    const bool euclid = a.metric == NK_METRIC_EUCLIDEAN;
    const int P = simt_cap_for_k(a.k);
    const size_t smem_budget = 96 * 1024;  // keeps >= 2 CTAs per SM
    const uint32_t num_iv = (a.n + SIMT_RT - 1) / SIMT_RT;

    const uint32_t max_grid = (uint32_t)di.num_sms * 8;
    (void)esz;

    uint32_t grid_used = 0;
    if (a.ev_begin) NK_CUDA_OK(cudaEventRecord(a.ev_begin, a.stream));
    for (uint32_t q0 = 0; q0 < a.Q;) {
        uint32_t left = a.Q - q0;
        int qt = left >= 5 ? 8 : left >= 3 ? 4 : left == 2 ? 2 : 1;
        if (!vec) qt = left >= 3 ? 4 : 1;
        while (qt > 1 && (size_t)P * 8 + (size_t)qt * a.dim * 4 > smem_budget) qt = vec ? qt / 2 : 1;
        size_t smem = (size_t)P * 8 + (size_t)qt * a.dim * 4;
        if (smem > di.max_smem_optin) {
            set_error("dim=%u too large for the SIMT scan (needs %zu B shared memory)", a.dim, smem);
            return -1;
        }
        SimtKernel kern = pick_kernel(a.dtype, vec, euclid, qt);
        if (simt_ensure(reinterpret_cast<const void *>(kern), di.device_id, smem)) return -1;
        int occ = simt_occupancy(reinterpret_cast<const void *>(kern), di.device_id, smem);
        // One grid for every query group of this search so the per-CTA partial lists line up.
        if (grid_used == 0) {
            grid_used = (uint32_t)di.num_sms * (uint32_t)occ;
            if (grid_used > num_iv) grid_used = num_iv;
            if (grid_used > max_grid) grid_used = max_grid;
            if (ws_reserve((void **)&ws.cand, &ws.cand_bytes, (size_t)grid_used * 8 * P * 8)) return -1;
            if (ws_reserve((void **)&ws.partial, &ws.partial_bytes, (size_t)a.Q * grid_used * a.k * 8)) return -1;
        }
        SimtParams p;
        p.rows = a.rows; p.n = a.n; p.dim = a.dim; p.row_base = a.row_base;
        p.queries = a.queries; p.q0 = q0; p.nq = left < (uint32_t)qt ? left : (uint32_t)qt; p.k = a.k;
        p.metric = a.metric; p.P = P; p.cand = ws.cand; p.partial = ws.partial; p.flags = ws.flags; p.only_if = a.only_if; p.below = a.below; p.mask = a.row_mask; p.min_score = a.min_score;
        NK_CUDA_OK(launch_pdl(kern, dim3(grid_used), dim3(SIMT_THREADS), smem, a.stream, a.only_if != nullptr && !a.defer_tail, p));
        if (launches) ++*launches;
        if (a.main_launches) ++*a.main_launches;
        q0 += p.nq;
    }
    if (a.ev_end) NK_CUDA_OK(cudaEventRecord(a.ev_end, a.stream));
    // Fold the per-CTA lists: list l of query q starts at partial[(q*grid + l)*k].
    // ... and, when the caller wants them, the decoded (index, score) arrays in the same launch
    if (merge_keys(ws.partial, grid_used, a.k, (size_t)grid_used * a.k, a.Q, a.k, out_keys, a.stream, a.only_if, 0, a.out_idx, a.out_score,
                   a.metric))
        return -1;
    if (launches) ++*launches;
    return 0;
}

}  // namespace nk
