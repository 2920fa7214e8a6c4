// cluster_search.cu — cluster-routed exact search (ClusterIndex.SearchWithClusters, pkg/gpu/kmeans.go:816-836) for a batch
// of queries, device-resident from routing to the decoded result.
//
// Layout (built once by nk_index_set_clusters, counting sort on the device): centroids [K x dim], CSR offsets [K+1] and the
// member rows sorted by (cluster, row).  Rows are read IN PLACE through the member list; there is no permuted copy.
//
// One search (per chunk of queries) is five launches:
//   route   Q x K squared distances (fp32 differences, fp64 squares: squaredEuclidean, kmeans.go:430-454), then the last
//           CTA of each query group ranks its queries' keys (distance asc, id asc) and writes the P nearest ids;
//   bucket  one CTA inverts the probe lists into each cluster's list of probing queries, and lays out the work list: per
//           cluster, ceil(queries / QT) chunks times ceil(rows / RR) row ranges, the chunks of one range next to each
//           other so that a cluster probed by more than QT queries is read from HBM once and from L2 afterwards;
//   scan    persistent CUDA-core kernel over the work list: the inner loop of knn_scan_simt_kernel (queries in shared
//           memory, 16-byte row loads, butterfly reduce-scatter, per-(CTA, query) candidate buffer with warp prunes, row
//           mask and score floor inside), rows addressed through the member list;  each (item, query) emits its best k;
//   merge   merge_keys over each query's own lists;
//   decode  key -> (row, score).  Keys carry ~(position in the query's candidate list) in the low word, so exact ties go
//           to the earlier position: probe rank first, then ascending row — the order GetClusterMembers + SearchCandidates
//           (kmeans.go:839-895) see.
#include <algorithm>

#include "simt_lane.cuh"
#include "scan_tensor_shared.cuh"

namespace nk {

int simt_cap_for_k(uint32_t k);

constexpr int CS_THREADS = 256;
constexpr int CS_WARPS = CS_THREADS / 32;
constexpr int CS_RT = 256;             // rows a CTA scores between two prune checks (as SIMT_RT)
constexpr int RT_QB = 4;               // queries per route CTA (centroid rows re-used from registers)
constexpr int RT_CPB = 64;             // centroids per route CTA
constexpr int BK_THREADS = 1024;       // bucket kernel (one CTA)
constexpr uint32_t LAYOUT_TILE = 8192; // rows per tile of the layout's counting sort
constexpr size_t PARTIAL_BUDGET = 256ull << 20;  // per-(item, query) lists of one chunk of queries
constexpr uint64_t LIST_KEYS = 4ull << 20;  // per-(item, query) list keys of one search the ranges may add up to

void ClusterLayout::release() {
    void *ptrs[] = {centroids, offs, members, build};
    for (void *q : ptrs)
        if (q) cudaFree(q);
    *this = ClusterLayout();
}

int ClusterSearchWs::release() {
    void *ptrs[] = {arena, counters, cand};
    for (void *q : ptrs)
        if (q) cudaFree(q);
    *this = ClusterSearchWs();
    return 0;
}

// Exclusive scan of one value per thread across the CTA (blockDim.x a multiple of 32).  *total = sum over the CTA.
__device__ __forceinline__ uint32_t cta_excl_scan(uint32_t v, uint32_t *s_warp, uint32_t *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    uint32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const uint32_t w = lane < nw ? s_warp[lane] : 0u;
        uint32_t wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        if (lane < nw) s_warp[lane] = wi - w;
        if (lane == 31) s_warp[32] = wi;
    }
    __syncthreads();
    const uint32_t r = s_warp[warp] + incl - v;
    *total = s_warp[32];
    return r;
}

// ---- layout: stable counting sort of the rows by cluster -----------------------------------------------------------------
__global__ void __launch_bounds__(256) layout_count_kernel(const int32_t *assign, uint64_t n, uint32_t K, uint32_t ntiles, uint32_t *tilecnt) {
    extern __shared__ uint32_t hist[];
    for (uint32_t c = threadIdx.x; c < K; c += blockDim.x) hist[c] = 0;
    __syncthreads();
    const uint64_t lo = (uint64_t)blockIdx.x * LAYOUT_TILE, hi = min(n, lo + LAYOUT_TILE);
    for (uint64_t r = lo + threadIdx.x; r < hi; r += blockDim.x) {
        const int32_t c = assign[r];
        if (c >= 0 && (uint32_t)c < K) atomicAdd(&hist[c], 1u);
    }
    __syncthreads();
    for (uint32_t c = threadIdx.x; c < K; c += blockDim.x) tilecnt[(size_t)c * ntiles + blockIdx.x] = hist[c];
}

// In place exclusive scan of tilecnt [K][ntiles] (cluster-major): entry (c, t) becomes the first output slot of tile t's
// members of cluster c.  offs[c] = the entry (c, 0), offs[K] = rows assigned.
__global__ void __launch_bounds__(1024) layout_scan_kernel(uint32_t *tilecnt, uint32_t K, uint32_t ntiles, uint32_t *offs) {
    __shared__ uint32_t s_warp[33];
    const size_t total = (size_t)K * ntiles;
    uint32_t carry = 0;
    for (size_t base = 0; base < total; base += blockDim.x) {
        const size_t i = base + threadIdx.x;
        const uint32_t v = i < total ? tilecnt[i] : 0u;
        uint32_t sum;
        const uint32_t ex = cta_excl_scan(v, s_warp, &sum) + carry;
        if (i < total) {
            tilecnt[i] = ex;
            if (i % ntiles == 0) offs[i / ntiles] = ex;
        }
        carry += sum;
    }
    if (threadIdx.x == 0) offs[K] = carry;
}

// One warp per tile walks its rows in order: peers of the same cluster in a 32-row step are ranked by lane, so members end
// up sorted by (cluster, row).
__global__ void __launch_bounds__(32) layout_scatter_kernel(const int32_t *assign, uint64_t n, uint32_t K, uint32_t ntiles,
                                                            const uint32_t *tilecnt, uint32_t *members) {
    extern __shared__ uint32_t run[];
    const int lane = threadIdx.x;
    for (uint32_t c = lane; c < K; c += 32) run[c] = 0;
    __syncwarp();
    const uint64_t lo = (uint64_t)blockIdx.x * LAYOUT_TILE, hi = min(n, lo + LAYOUT_TILE);
    for (uint64_t r0 = lo; r0 < hi; r0 += 32) {
        const uint64_t r = r0 + lane;
        int32_t c = r < hi ? assign[r] : -1;
        if (c < 0 || (uint32_t)c >= K) c = -1;
        const uint32_t peers = __match_any_sync(0xffffffffu, c);
        const uint32_t rank = __popc(peers & ((1u << lane) - 1u));
        uint32_t base = 0;
        if (c >= 0) {
            base = run[c];
            members[tilecnt[(size_t)c * ntiles + blockIdx.x] + base + rank] = (uint32_t)r;
        }
        __syncwarp();
        if (c >= 0 && rank == 0) run[c] = base + __popc(peers);
        __syncwarp();
    }
}

int cluster_layout_build(ClusterLayout &L, const float *centroids_host, uint32_t K, uint32_t dim, const int32_t *assign_host,
                         uint64_t n_rows, cudaStream_t s, uint64_t *launches) {
    L.on = false;
    const uint32_t ntiles = (uint32_t)((n_rows + LAYOUT_TILE - 1) / LAYOUT_TILE);
    const size_t a_bytes = (n_rows * 4 + 255) & ~(size_t)255, t_bytes = (size_t)K * (ntiles ? ntiles : 1) * 4;
    if (ws_reserve((void **)&L.centroids, &L.centroids_bytes, (size_t)K * dim * 4)) return -1;
    if (ws_reserve((void **)&L.offs, &L.offs_bytes, (size_t)(K + 1) * 4)) return -1;
    if (ws_reserve((void **)&L.members, &L.members_bytes, (size_t)(n_rows ? n_rows : 1) * 4)) return -1;
    if (ws_reserve(&L.build, &L.build_bytes, a_bytes + t_bytes)) return -1;
    int32_t *d_assign = static_cast<int32_t *>(L.build);
    uint32_t *tilecnt = reinterpret_cast<uint32_t *>(static_cast<unsigned char *>(L.build) + a_bytes);
    NK_CUDA_OK(cudaMemcpyAsync(L.centroids, centroids_host, (size_t)K * dim * 4, cudaMemcpyHostToDevice, s));
    if (n_rows) NK_CUDA_OK(cudaMemcpyAsync(d_assign, assign_host, n_rows * 4, cudaMemcpyHostToDevice, s));
    if (ntiles) {
        layout_count_kernel<<<ntiles, 256, (size_t)K * 4, s>>>(d_assign, n_rows, K, ntiles, tilecnt);
        NK_CUDA_OK(cudaGetLastError());
        layout_scan_kernel<<<1, 1024, 0, s>>>(tilecnt, K, ntiles, L.offs);
        NK_CUDA_OK(cudaGetLastError());
        layout_scatter_kernel<<<ntiles, 32, (size_t)K * 4, s>>>(d_assign, n_rows, K, ntiles, tilecnt, L.members);
        NK_CUDA_OK(cudaGetLastError());
        if (launches) *launches += 3;
    } else {
        NK_CUDA_OK(cudaMemsetAsync(L.offs, 0, (size_t)(K + 1) * 4, s));
    }
    std::vector<uint32_t> offs(K + 1);
    NK_CUDA_OK(cudaMemcpyAsync(offs.data(), L.offs, (size_t)(K + 1) * 4, cudaMemcpyDeviceToHost, s));
    NK_CUDA_OK(cudaStreamSynchronize(s));
    uint32_t mx = 0;
    for (uint32_t c = 0; c < K; ++c) mx = std::max(mx, offs[c + 1] - offs[c]);
    L.K = K; L.max_rows = mx; L.n_assigned = offs[K]; L.on = true;
    return 0;
}

// ---- route ------------------------------------------------------------------------------------------------------------
struct RouteParams {
    const float *queries;  // chunk base
    uint32_t Q, dim;
    const float *cen;
    uint32_t K, P;
    uint64_t *dist;  // [Q][K] keys (ord(-distance) << 32 | ~id)
    int *counters;   // [ceil(Q / RT_QB)]
    int32_t *probe;  // [Q][P]
    int32_t *out_probe;  // nullable, [Q][P]
};

__global__ void __launch_bounds__(CS_THREADS) cluster_route_kernel(RouteParams p) {
    extern __shared__ uint64_t sk[];  // [K] keys of one query (last CTA of the group only)
    __shared__ int s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t q0 = blockIdx.y * RT_QB, nq = min((uint32_t)RT_QB, p.Q - q0), dim = p.dim;
    const uint32_t c_end = min(p.K, (blockIdx.x + 1) * RT_CPB);
    for (uint32_t c = blockIdx.x * RT_CPB + warp; c < c_end; c += CS_WARPS) {
        double acc[RT_QB];
#pragma unroll
        for (int i = 0; i < RT_QB; ++i) acc[i] = 0.0;
        const float *cp = p.cen + (size_t)c * dim;
        for (uint32_t j = lane; j < dim; j += 32) {
            const float cv = __ldg(cp + j);
#pragma unroll
            for (int i = 0; i < RT_QB; ++i)
                if ((uint32_t)i < nq) {
                    const float d = __ldg(p.queries + (size_t)(q0 + i) * dim + j) - cv;  // float32 difference, float64 square
                    acc[i] = fma((double)d, (double)d, acc[i]);
                }
        }
#pragma unroll
        for (int i = 0; i < RT_QB; ++i)
#pragma unroll
            for (int o = 16; o; o >>= 1) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
        if (lane == 0) {
#pragma unroll
            for (int i = 0; i < RT_QB; ++i)
                if ((uint32_t)i < nq) p.dist[(size_t)(q0 + i) * p.K + c] = make_key(-(float)acc[i], c);
        }
    }
    // the last CTA of this query group to finish selects the P nearest centroids of each of its queries
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(&p.counters[blockIdx.y], 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (uint32_t i = 0; i < nq; ++i) {
        const uint32_t q = q0 + i;
        for (uint32_t c = tid; c < p.K; c += CS_THREADS) sk[c] = __ldcg(p.dist + (size_t)q * p.K + c);
        __syncthreads();
        // rank = number of better keys (keys are distinct: the id is in the low word); stop counting at P
        for (uint32_t c = tid; c < p.K; c += CS_THREADS) {
            const uint64_t key = sk[c];
            uint32_t better = 0;
            for (uint32_t j = 0; j < p.K && better < p.P; ++j) better += sk[j] > key ? 1u : 0u;
            if (better < p.P) {
                p.probe[(size_t)q * p.P + better] = (int32_t)c;
                if (p.out_probe) p.out_probe[(size_t)q * p.P + better] = (int32_t)c;
            }
        }
        __syncthreads();
    }
    if (tid == 0) p.counters[blockIdx.y] = 0;  // ready for the next search
}

// ---- bucket -----------------------------------------------------------------------------------------------------------
struct BucketParams {
    const int32_t *probe;  // [Q][P]
    uint32_t Q, P, K, QT, RR;
    const uint32_t *offs;  // [K+1]
    uint32_t *qcnt, *qoff;  // [K] probing queries per cluster, offset of its list in qlist
    uint32_t *item_off;     // [K+1] first work item of each cluster; item_off[K] = number of items
    uint32_t *qlist;        // [Q*P] probe entries (q * P + r) grouped by cluster
    uint32_t *base_pos;     // [Q*P] position of the probe's first member in the query's candidate list
    uint32_t *slot_off;     // [Q*P] first partial list of the probe's ranges
    uint32_t *nslots;       // [Q] partial lists of the query
};

__global__ void __launch_bounds__(BK_THREADS) cluster_bucket_kernel(BucketParams p) {
    extern __shared__ uint32_t sm[];  // cnt[K], fill[K]
    __shared__ uint32_t s_warp[33];
    uint32_t *cnt = sm, *fill = sm + p.K;
    const uint32_t tid = threadIdx.x, E = p.Q * p.P;
    for (uint32_t c = tid; c < p.K; c += BK_THREADS) cnt[c] = 0;
    __syncthreads();
    for (uint32_t e = tid; e < E; e += BK_THREADS) atomicAdd(&cnt[p.probe[e]], 1u);
    __syncthreads();
    uint32_t qcarry = 0, icarry = 0;
    for (uint32_t base = 0; base < p.K; base += BK_THREADS) {
        const uint32_t c = base + tid;
        uint32_t nq = 0, items = 0;
        if (c < p.K) {
            nq = cnt[c];
            const uint32_t m = p.offs[c + 1] - p.offs[c];
            items = nq ? ((nq + p.QT - 1) / p.QT) * ((m + p.RR - 1) / p.RR) : 0u;
        }
        uint32_t qs, is;
        const uint32_t qx = cta_excl_scan(nq, s_warp, &qs) + qcarry;
        const uint32_t ix = cta_excl_scan(items, s_warp, &is) + icarry;
        if (c < p.K) {
            fill[c] = qx;
            p.qcnt[c] = nq; p.qoff[c] = qx; p.item_off[c] = ix;
        }
        qcarry += qs; icarry += is;
    }
    if (tid == 0) p.item_off[p.K] = icarry;
    __syncthreads();
    for (uint32_t e = tid; e < E; e += BK_THREADS) p.qlist[atomicAdd(&fill[p.probe[e]], 1u)] = e;
    for (uint32_t q = tid; q < p.Q; q += BK_THREADS) {
        uint32_t pos = 0, sl = 0;
        for (uint32_t r = 0; r < p.P; ++r) {
            const uint32_t e = q * p.P + r, c = (uint32_t)p.probe[e], m = p.offs[c + 1] - p.offs[c];
            p.base_pos[e] = pos;
            p.slot_off[e] = sl;
            pos += m;
            sl += (m + p.RR - 1) / p.RR;
        }
        p.nslots[q] = sl;
    }
}

// ---- scan -------------------------------------------------------------------------------------------------------------
struct CScanParams {
    const void *rows;
    uint32_t dim, P, k;
    int metric;
    const float *queries;  // chunk base
    int Pc;                // candidate-buffer capacity (power of two)
    uint64_t *cand;        // [grid][QT][Pc]
    uint64_t *partial;     // [Q][slots_max][k]
    uint32_t slots_max;
    int *flags;
    const uint32_t *mask;
    float min_score;
    const uint32_t *offs, *members;
    uint32_t K, RR;
    const uint32_t *qcnt, *qoff, *item_off, *qlist, *base_pos, *slot_off;
};

template <typename T, bool VEC, int QT, int R, bool EUCLID>
__global__ void __launch_bounds__(CS_THREADS) cluster_scan_kernel(CScanParams p) {
    using L = Lane<T, VEC>;
    constexpr int EPL = L::EPL;
    constexpr int CH = 32 * EPL;
    constexpr int V = R * QT;
    static_assert(V <= 32 && (32 % V) == 0, "R*QT must divide 32");
    constexpr int LPV = 32 / V;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *sbuf = reinterpret_cast<uint64_t *>(smem_raw);
    float *qs = reinterpret_cast<float *>(smem_raw + (size_t)p.Pc * 8);  // [QT][dim]
    __shared__ float s_qq[QT];
    __shared__ float s_tau[QT];
    __shared__ int s_cnt[QT];
    __shared__ uint32_t s_e[QT], s_pos0[QT];
    __shared__ uint32_t s_rid[CS_RT];  // member rows of the current interval
    __shared__ uint32_t s_c, s_rho, s_nq;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t dim = p.dim;
    const T *rows = static_cast<const T *>(p.rows);
    uint64_t *my_cand = p.cand + (size_t)blockIdx.x * QT * p.Pc;
    const int prune_at = p.Pc - CS_RT;
    const uint32_t nsteps = (dim + CH - 1) / CH;
    const uint32_t n_items = p.item_off[p.K];

    for (uint32_t it = blockIdx.x; it < n_items; it += gridDim.x) {
        if (tid == 0) {
            uint32_t lo = 0, hi = p.K;  // last cluster c with item_off[c] <= it
            while (hi - lo > 1) {
                const uint32_t mid = (lo + hi) >> 1;
                if (p.item_off[mid] <= it) lo = mid;
                else hi = mid;
            }
            const uint32_t c = lo, chunks = (p.qcnt[c] + QT - 1) / QT, local = it - p.item_off[c];
            const uint32_t chi = local % chunks;
            s_c = c; s_rho = local / chunks;
            s_nq = min((uint32_t)QT, p.qcnt[c] - chi * QT);
            for (uint32_t i = 0; i < s_nq; ++i) {
                const uint32_t e = p.qlist[p.qoff[c] + chi * QT + i];
                s_e[i] = e;
                s_pos0[i] = p.base_pos[e];
            }
        }
        __syncthreads();
        const uint32_t c = s_c, rho = s_rho, nq = s_nq;
        const uint32_t m_lo = p.offs[c] + rho * p.RR, m_hi = min(p.offs[c + 1], m_lo + p.RR), pos_c = p.offs[c];
        for (uint32_t i = tid; i < (uint32_t)QT * dim; i += CS_THREADS) {
            const uint32_t qi = i / dim, j = i - qi * dim;
            qs[i] = qi < nq ? p.queries[(size_t)(s_e[qi] / p.P) * dim + j] : 0.0f;
        }
        if (tid < QT) {
            s_tau[tid] = p.min_score;
            s_cnt[tid] = 0;
        }
        __syncthreads();
        for (int qi = warp; qi < QT; qi += CS_WARPS) {
            float a = 0.0f;
            for (uint32_t j = lane; j < dim; j += 32) a = fmaf(qs[qi * dim + j], qs[qi * dim + j], a);
#pragma unroll
            for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if (lane == 0) s_qq[qi] = a;
        }
        __syncthreads();

        for (uint32_t base = m_lo; base < m_hi; base += CS_RT) {
            if (tid < CS_RT) s_rid[tid] = base + tid < m_hi ? __ldg(p.members + base + tid) : 0u;
            __syncthreads();
#pragma unroll 1
            for (int t = 0; t < CS_RT / (CS_WARPS * R); ++t) {
                const uint32_t m0 = base + (uint32_t)(t * CS_WARPS + warp) * R;
                if (m0 >= m_hi) continue;  // warp-uniform
                const T *rp[R];
                uint32_t rid[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const uint32_t mm = m0 + r < m_hi ? m0 + r : m_hi - 1;  // clamp; masked below
                    rid[r] = s_rid[mm - base];
                    rp[r] = rows + (size_t)rid[r] * dim;
                }
                float acc[V];
                float xx[R];
#pragma unroll
                for (int i = 0; i < V; ++i) acc[i] = 0.0f;
#pragma unroll
                for (int r = 0; r < R; ++r) xx[r] = 0.0f;

#pragma unroll 2
                for (uint32_t cs = 0; cs < nsteps; ++cs) {
                    const uint32_t e = cs * CH + lane * EPL;
                    if (e < dim) {
                        float x[R][EPL];
#pragma unroll
                        for (int r = 0; r < R; ++r) L::load(rp[r] + e, x[r]);
#pragma unroll
                        for (int qi = 0; qi < QT; ++qi) {
                            if ((uint32_t)qi >= nq) continue;  // CTA-uniform: a chunk of fewer queries does fewer FMAs
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

                warp_reduce_scatter<V>(acc, lane);
                const int j = lane / LPV;
                const int r = j / QT, qi = j - r * QT;
                float s = acc[0];
                float xr = 0.0f;
                if constexpr (!EUCLID) {
                    warp_reduce_scatter<R>(xx, lane);
                    xr = __shfl_sync(0xffffffffu, xx[0], r * (32 / R));
                }
                uint32_t row = rid[0];
#pragma unroll
                for (int rr = 1; rr < R; ++rr)
                    if (rr == r) row = rid[rr];
                const uint32_t m = m0 + r;
                if ((lane % LPV) == 0 && m < m_hi && (uint32_t)qi < nq && (!p.mask || ((p.mask[row >> 5] >> (row & 31)) & 1u))) {
                    if constexpr (EUCLID) {
                        s = -s;
                    } else if (p.metric == NK_METRIC_COSINE) {
                        float den = sqrtf(xr * s_qq[qi]);
                        s = den > 0.0f ? s / den : 0.0f;
                    }
                    if (s != s) s = -INFINITY;
                    if (s >= s_tau[qi] && s >= p.min_score) {
                        const uint64_t key = make_key(s, s_pos0[qi] + (m - pos_c));
                        int pos = atomicAdd(&s_cnt[qi], 1);
                        if (pos < p.Pc) my_cand[(size_t)qi * p.Pc + pos] = key;
                        else atomicExch(p.flags, 1);
                    }
                }
            }
            __syncthreads();
            uint32_t need = 0;
#pragma unroll
            for (int qi = 0; qi < QT; ++qi) need |= (s_cnt[qi] > prune_at ? 1u : 0u) << qi;
            __syncthreads();
            if (need && p.Pc == 512) {
                if (warp < QT && (need & (1u << warp)))
                    warp_prune<16>(my_cand + (size_t)warp * p.Pc, &s_cnt[warp], &s_tau[warp], p.k, lane, nullptr, 0, false, 0.0f, (int)p.k, p.min_score);
                __syncthreads();
            } else if (need) {
#pragma unroll 1
                for (int qi = 0; qi < QT; ++qi)
                    if (need & (1u << qi)) block_prune(my_cand + (size_t)qi * p.Pc, p.Pc, &s_cnt[qi], &s_tau[qi], p.k, sbuf, p.Pc);
            }
        }

        // emit this item's best k per query into the query's list for (probe, range)
        __syncthreads();
        if (p.Pc == 512) {
            for (uint32_t qi = warp; qi < nq; qi += CS_WARPS) {
                const uint32_t e = s_e[qi];
                uint64_t *dst = p.partial + ((size_t)(e / p.P) * p.slots_max + p.slot_off[e] + rho) * p.k;
                warp_prune<16>(my_cand + (size_t)qi * p.Pc, &s_cnt[qi], &s_tau[qi], p.k, lane, dst, (int)p.k, false, 0.0f, (int)p.k, p.min_score);
            }
        } else {
#pragma unroll 1
            for (uint32_t qi = 0; qi < nq; ++qi) {
                block_prune(my_cand + (size_t)qi * p.Pc, p.Pc, &s_cnt[qi], &s_tau[qi], p.k, sbuf, p.Pc);
                const uint32_t e = s_e[qi];
                uint64_t *dst = p.partial + ((size_t)(e / p.P) * p.slots_max + p.slot_off[e] + rho) * p.k;
                for (uint32_t i = tid; i < p.k; i += CS_THREADS) dst[i] = sbuf[i];
            }
        }
        __syncthreads();
    }
}

// ---- decode -----------------------------------------------------------------------------------------------------------
__global__ void cluster_decode_kernel(const uint64_t *keys, uint32_t Q, uint32_t k, uint32_t P, const int32_t *probe, const uint32_t *base_pos,
                                      const uint32_t *offs, const uint32_t *members, uint64_t row_base, int metric, uint32_t *out_idx,
                                      float *out_score) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)Q * k) return;
    const uint64_t key = keys[i];
    if (!key) {
        out_idx[i] = 0xffffffffu;
        out_score[i] = 0.0f;
        return;
    }
    const uint32_t q = (uint32_t)(i / k), pos = key_row(key);
    const uint32_t *bp = base_pos + (size_t)q * P;
    uint32_t lo = 0, hi = P;  // last probe whose first position is <= pos (an empty cluster shares its successor's)
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (bp[mid] <= pos) lo = mid;
        else hi = mid;
    }
    const uint32_t c = (uint32_t)probe[(size_t)q * P + lo];
    float s = key_score(key);
    if (metric == NK_METRIC_EUCLIDEAN) s = sqrtf(fmaxf(-s, 0.0f));
    out_idx[i] = (uint32_t)(row_base + members[offs[c] + pos - bp[lo]]);
    out_score[i] = s;
}

// ---------------------------------------------------------------------------------------------------------------------
typedef void (*CScanKernel)(CScanParams);

template <typename T, bool VEC, bool EUCLID>
static CScanKernel pick_cs_qt(int qt) {
    return qt == 8 ? cluster_scan_kernel<T, VEC, 8, 4, EUCLID> : cluster_scan_kernel<T, VEC, 1, 8, EUCLID>;
}
static CScanKernel pick_cs_kernel(int dtype, bool vec, bool euclid, int qt) {
    if (dtype == NK_DTYPE_F16) {
        if (vec) return euclid ? pick_cs_qt<__half, true, true>(qt) : pick_cs_qt<__half, true, false>(qt);
        return euclid ? pick_cs_qt<__half, false, true>(qt) : pick_cs_qt<__half, false, false>(qt);
    }
    if (dtype == NK_DTYPE_BF16) {
        if (vec) return euclid ? pick_cs_qt<__nv_bfloat16, true, true>(qt) : pick_cs_qt<__nv_bfloat16, true, false>(qt);
        return euclid ? pick_cs_qt<__nv_bfloat16, false, true>(qt) : pick_cs_qt<__nv_bfloat16, false, false>(qt);
    }
    if (vec) return euclid ? pick_cs_qt<float, true, true>(qt) : pick_cs_qt<float, true, false>(qt);
    return euclid ? pick_cs_qt<float, false, true>(qt) : pick_cs_qt<float, false, false>(qt);
}

static size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

int cluster_search(const DeviceInfo &di, const ClusterLayout &L, const ClusterSearchArgs &a, ClusterSearchWs &ws, uint64_t *launches) {
    if (!L.on) { set_error("no clusters set (nk_index_set_clusters)"); return -1; }
    if (a.Q == 0 || a.k == 0) return 0;
    if (a.k > NK_MAX_K) { set_error("k=%u exceeds NK_MAX_K=%u", a.k, NK_MAX_K); return -1; }
    const uint32_t K = L.K, P = std::min(a.n_probe, K), k = a.k, dim = a.dim;
    const bool vec = (dim % (a.dtype == NK_DTYPE_F32 ? 4u : 8u) == 0) && ((reinterpret_cast<uintptr_t>(a.rows) & 15) == 0);
    const bool euclid = a.metric == NK_METRIC_EUCLIDEAN;
    const int Pc = simt_cap_for_k(k);
    // 8 queries per work item while two CTAs fit an SM, else one (very wide rows)
    int qt = 8;
    size_t smem = (size_t)Pc * 8 + (size_t)qt * dim * 4;
    if (smem > 113 * 1024) { qt = 1; smem = (size_t)Pc * 8 + (size_t)dim * 4; }
    if (smem > di.max_smem_optin) { set_error("dim=%u too large for the cluster scan (needs %zu B shared memory)", dim, smem); return -1; }
    if ((size_t)K * 8 > di.max_smem_optin) { set_error("K=%u too large", K); return -1; }
    CScanKernel kern = pick_cs_kernel(a.dtype, vec, euclid, qt);
    NK_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    NK_CUDA_OK(cudaFuncSetAttribute(cluster_route_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(K * 8)));
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, CS_THREADS, smem) != cudaSuccess) { cudaGetLastError(); occ = 1; }
    occ = std::max(1, std::min(occ, 8));
    const uint32_t grid = (uint32_t)di.num_sms * (uint32_t)occ;

    // Plan: rows per range RR (enough work items to fill the grid, at most maxr_cap ranges per cluster and a per-query list
    // block within the budget), and the query chunk Qc that keeps the partial lists within PARTIAL_BUDGET.
    const uint64_t m_avg = std::max<uint64_t>(1, L.n_assigned / K);
    const uint32_t max_rows = std::max<uint32_t>(1, L.max_rows);
    // ranges per cluster: many for small batches (one hot cluster must not serialise the grid), few for large ones (the
    // lists of every (range, query) are merged)
    const uint64_t maxr_cap = std::max<uint64_t>(1, std::min<uint64_t>({4096, std::max<uint64_t>(16, LIST_KEYS / ((uint64_t)a.Q * P * k)),
                                                                        PARTIAL_BUDGET / ((uint64_t)P * k * 8)}));
    uint32_t Qc = a.Q, RR = 0, slots_max = 0;
    for (int pass = 0; pass < 3; ++pass) {
        const uint64_t probes = (uint64_t)Qc * P;
        const uint64_t sharing = std::max<uint64_t>(1, std::min<uint64_t>(qt, probes / K));
        const uint64_t chunks = (probes + sharing - 1) / sharing;
        uint64_t rr = (m_avg * chunks + 4ull * grid - 1) / (4ull * grid);
        rr = std::max<uint64_t>(rr, 64);
        rr = std::max<uint64_t>(rr, (max_rows + maxr_cap - 1) / maxr_cap);
        rr = (rr + 31) / 32 * 32;
        RR = (uint32_t)std::min<uint64_t>(rr, 0x40000000ull);
        slots_max = P * ((max_rows + RR - 1) / RR);
        const size_t per_q = (size_t)slots_max * k * 8;
        const uint32_t fit = (uint32_t)std::max<size_t>(1, PARTIAL_BUDGET / per_q);
        if (fit >= Qc) break;
        Qc = fit;
    }
    const uint32_t QG = (Qc + RT_QB - 1) / RT_QB;

    // workspace (grow-only): carve the arena
    const size_t b_dist = al256((size_t)Qc * K * 8), b_probe = al256((size_t)Qc * P * 4), b_k = al256((size_t)K * 4),
                 b_k1 = al256((size_t)(K + 1) * 4), b_q = al256((size_t)Qc * 4), b_part = al256((size_t)Qc * slots_max * k * 8),
                 b_keys = al256((size_t)Qc * k * 8);
    const size_t need = b_dist + b_probe * 4 + b_k * 2 + b_k1 + b_q + b_part + b_keys;
    if (ws_reserve(&ws.arena, &ws.arena_bytes, need)) return -1;
    {
        void *old = ws.counters;
        const size_t old_bytes = ws.counters_bytes;
        if (ws_reserve((void **)&ws.counters, &ws.counters_bytes, (size_t)QG * 4)) return -1;
        if (ws.counters != old || ws.counters_bytes != old_bytes) NK_CUDA_OK(cudaMemsetAsync(ws.counters, 0, ws.counters_bytes, a.stream));
    }
    if (ws_reserve((void **)&ws.cand, &ws.cand_bytes, (size_t)grid * qt * Pc * 8)) return -1;
    unsigned char *cur = static_cast<unsigned char *>(ws.arena);
    auto take = [&](size_t b) { unsigned char *r = cur; cur += b; return r; };
    uint64_t *dist = reinterpret_cast<uint64_t *>(take(b_dist));
    int32_t *probe = reinterpret_cast<int32_t *>(take(b_probe));
    uint32_t *qlist = reinterpret_cast<uint32_t *>(take(b_probe));
    uint32_t *base_pos = reinterpret_cast<uint32_t *>(take(b_probe));
    uint32_t *slot_off = reinterpret_cast<uint32_t *>(take(b_probe));
    uint32_t *qcnt = reinterpret_cast<uint32_t *>(take(b_k));
    uint32_t *qoff = reinterpret_cast<uint32_t *>(take(b_k));
    uint32_t *item_off = reinterpret_cast<uint32_t *>(take(b_k1));
    uint32_t *nslots = reinterpret_cast<uint32_t *>(take(b_q));
    uint64_t *partial = reinterpret_cast<uint64_t *>(take(b_part));
    uint64_t *keys = reinterpret_cast<uint64_t *>(take(b_keys));

    for (uint32_t q0 = 0; q0 < a.Q; q0 += Qc) {
        const uint32_t nq = std::min(Qc, a.Q - q0);
        const float *qp = a.queries + (size_t)q0 * dim;
        RouteParams rp{qp, nq, dim, L.centroids, K, P, dist, ws.counters, probe, a.out_probe ? a.out_probe + (size_t)q0 * P : nullptr};
        cluster_route_kernel<<<dim3((K + RT_CPB - 1) / RT_CPB, (nq + RT_QB - 1) / RT_QB), CS_THREADS, (size_t)K * 8, a.stream>>>(rp);
        NK_CUDA_OK(cudaGetLastError());
        BucketParams bp{probe, nq, P, K, (uint32_t)qt, RR, L.offs, qcnt, qoff, item_off, qlist, base_pos, slot_off, nslots};
        cluster_bucket_kernel<<<1, BK_THREADS, (size_t)K * 8, a.stream>>>(bp);
        NK_CUDA_OK(cudaGetLastError());
        CScanParams sp;
        sp.rows = a.rows; sp.dim = dim; sp.P = P; sp.k = k; sp.metric = a.metric; sp.queries = qp; sp.Pc = Pc; sp.cand = ws.cand;
        sp.partial = partial; sp.slots_max = slots_max; sp.flags = a.flags; sp.mask = a.row_mask; sp.min_score = a.min_score;
        sp.offs = L.offs; sp.members = L.members; sp.K = K; sp.RR = RR; sp.qcnt = qcnt; sp.qoff = qoff; sp.item_off = item_off;
        sp.qlist = qlist; sp.base_pos = base_pos; sp.slot_off = slot_off;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        if (a.timing) {
            NK_CUDA_OK(cudaEventCreate(&e0));
            NK_CUDA_OK(cudaEventCreate(&e1));
            NK_CUDA_OK(cudaEventRecord(e0, a.stream));
        }
        kern<<<grid, CS_THREADS, smem, a.stream>>>(sp);
        NK_CUDA_OK(cudaGetLastError());
        if (a.timing) {
            NK_CUDA_OK(cudaEventRecord(e1, a.stream));
            a.timing_events->emplace_back(e0, e1);
        }
        if (merge_keys(partial, slots_max, k, (size_t)slots_max * k, nq, k, keys, a.stream, nullptr, 0, nullptr, nullptr, 0, nullptr, 0,
                       nullptr, nslots))
            return -1;
        const size_t total = (size_t)nq * k;
        cluster_decode_kernel<<<(unsigned)((total + 255) / 256), 256, 0, a.stream>>>(keys, nq, k, P, probe, base_pos, L.offs, L.members, a.row_base,
                                                                                     a.metric, a.out_idx + (size_t)q0 * k, a.out_score + (size_t)q0 * k);
        NK_CUDA_OK(cudaGetLastError());
        if (launches) *launches += 5;
    }
    return 0;
}

}  // namespace nk
