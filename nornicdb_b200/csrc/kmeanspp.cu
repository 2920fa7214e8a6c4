// kmeanspp.cu — k-means++ seeding over every row of an fp32 shard, on the device (initCentroidsKMeansPlusPlus,
// pkg/gpu/kmeans.go:364-427; DESIGN.md §3.8).
//
// One seeding step is three launches on the shard's stream:
//   update  persistent, CUDA cores: d2[i] <- min(d2[i], squaredEuclidean(row i, newest centroid)), strict <.  A row is
//           skipped unread when the triangle inequality proves the new centroid cannot be strictly closer:
//             d(c_near, c_new) >= 2 d(x, c_near)  =>  d(x, c_new) >= d(c_near, c_new) - d(x, c_near) >= d(x, c_near).
//           The test is cc[near[i]] >= 2 sqrt(d2[i]) (1 + 1e-5): squaredEuclidean rounds each float32 difference, so a
//           computed distance is within ~6e-8 (relative) of the exact one; the slack covers that with a wide margin, and
//           only when every value involved is finite.  Writes one fp64 sum of d2 per KPP_BLOCK rows in a fixed order.
//   select  one CTA: total = sum of the block sums, target = draw * total, the first block whose running offset plus
//           block sum reaches the target, then the first row of that block whose offset plus in-block prefix does (the
//           same `>=` at both levels; a block whose prefix falls short by rounding passes on to the next block).
//   cc      distances from the new centroid to every earlier one, by the same warp routine as the update.
#include <algorithm>
#include <limits.h>

#include "kernels.cuh"

namespace nk {
namespace {

constexpr int UPD_THREADS = 256;
constexpr int SEL_THREADS = KPP_BLOCK;  // one row per thread in the in-block scan
constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double acc4(double acc, float4 a, float4 b) {
    // float32 differences, float64 squares (squaredEuclidean, kmeans.go:430-454)
    double d = (double)(a.x - b.x); acc = fma(d, d, acc);
    d = (double)(a.y - b.y); acc = fma(d, d, acc);
    d = (double)(a.z - b.z); acc = fma(d, d, acc);
    d = (double)(a.w - b.w); return fma(d, d, acc);
}

// squaredEuclidean(x, c) by one warp; every lane returns the same total (butterfly reduction: both operands of each add
// are the same pair in either lane, so the result is bit-identical across lanes and runs).  STREAM: x is read once
// (corpus rows), c stays cached (a centroid).
template <bool STREAM>
__device__ __forceinline__ double warp_sq_euclid(const float *__restrict__ x, const float *__restrict__ c, uint32_t dim, bool vec4,
                                                 int lane) {
    double s0 = 0.0, s1 = 0.0;
    if (vec4) {
        const float4 *x4 = reinterpret_cast<const float4 *>(x), *c4 = reinterpret_cast<const float4 *>(c);
        const uint32_t d4 = dim / 4;
        uint32_t k = lane;
        for (; k + 96 < d4; k += 128) {  // four 16-byte loads in flight per lane
            float4 a0, a1, a2, a3;
            if (STREAM) { a0 = __ldcs(x4 + k); a1 = __ldcs(x4 + k + 32); a2 = __ldcs(x4 + k + 64); a3 = __ldcs(x4 + k + 96); }
            else { a0 = __ldg(x4 + k); a1 = __ldg(x4 + k + 32); a2 = __ldg(x4 + k + 64); a3 = __ldg(x4 + k + 96); }
            s0 = acc4(s0, a0, __ldg(c4 + k));
            s1 = acc4(s1, a1, __ldg(c4 + k + 32));
            s0 = acc4(s0, a2, __ldg(c4 + k + 64));
            s1 = acc4(s1, a3, __ldg(c4 + k + 96));
        }
        for (; k < d4; k += 32) s0 = acc4(s0, STREAM ? __ldcs(x4 + k) : __ldg(x4 + k), __ldg(c4 + k));
    } else {
        for (uint32_t k = lane; k < dim; k += 32) {
            const double d = (double)(__ldg(x + k) - __ldg(c + k));
            s0 = fma(d, d, s0);
        }
    }
    double s = s0 + s1;
#pragma unroll
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
    return s;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// Inclusive scan over the CTA in a fixed order (warp Hillis-Steele, then the warp totals); *total = the last prefix.
__device__ double cta_inclusive_scan(double v, double *warp_tot, double *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(FULL, v, o);
        if (lane >= o) v += u;
    }
    __syncthreads();  // warp_tot may still be read by a previous call
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double w = lane < nw ? warp_tot[lane] : 0.0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double u = __shfl_up_sync(FULL, w, o);
            if (lane >= o) w += u;
        }
        if (lane < nw) warp_tot[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v += warp_tot[warp - 1];
    *total = warp_tot[nw - 1];
    return v;
}

// Exclusive form of the same scan, by a shift rather than inclusive - own (inf - inf would be NaN).
__device__ double cta_exclusive_scan(double v, double *warp_tot, double *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const double incl = cta_inclusive_scan(v, warp_tot, total);
    const double prev = __shfl_up_sync(FULL, incl, 1);
    return lane > 0 ? prev : warp > 0 ? warp_tot[warp - 1] : 0.0;
}

__global__ void __launch_bounds__(UPD_THREADS) kpp_update_kernel(const float *__restrict__ rows, uint64_t n, uint32_t dim, bool vec4,
                                                                 const float *__restrict__ cen, uint32_t c, bool init,
                                                                 const double *__restrict__ cc, double *__restrict__ d2,
                                                                 int32_t *__restrict__ near, double *__restrict__ bsum,
                                                                 unsigned long long *scored) {
    __shared__ double tile_sum[KPP_BLOCK / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float *cn = cen + (size_t)c * dim;
    const uint64_t nblk = (n + KPP_BLOCK - 1) / KPP_BLOCK;
    unsigned long long my_scored = 0;
    for (uint64_t b = blockIdx.x; b < nblk; b += gridDim.x) {
        for (uint32_t t = warp; t < KPP_BLOCK / 32; t += UPD_THREADS / 32) {
            const uint64_t r0 = b * KPP_BLOCK + (uint64_t)t * 32, i = r0 + lane;
            const bool valid = i < n;
            double v = 0.0;
            int32_t nr = 0;
            bool need = valid;
            if (valid && !init) {
                v = d2[i];
                nr = near[i];
                const double dc = __ldg(cc + nr);
                if (isfinite(v) && isfinite(dc) && dc >= 2.0 * sqrt(v) * (1.0 + 1e-5)) need = false;
            }
            unsigned m = __ballot_sync(FULL, need);
            my_scored += lane == 0 ? __popc(m) : 0;
            bool changed = init && valid;
            while (m) {
                const int src = __ffs(m) - 1;
                m &= m - 1;
                const double dist = warp_sq_euclid<true>(rows + (r0 + src) * dim, cn, dim, vec4, lane);
                if (lane == src) {
                    if (init) v = dist;
                    else if (dist < v) { v = dist; nr = (int32_t)c; changed = true; }  // strict <, kmeans.go:414-421
                }
            }
            if (changed) { d2[i] = v; near[i] = nr; }
            const double s = warp_sum(v);
            if (lane == 0) tile_sum[t] = s;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int t = 0; t < (int)(KPP_BLOCK / 32); ++t) s += tile_sum[t];
            bsum[b] = s;
        }
        __syncthreads();
    }
    if (lane == 0 && my_scored) atomicAdd(scored, my_scored);
}

__global__ void __launch_bounds__(SEL_THREADS) kpp_select_kernel(int mode, const double *__restrict__ d2, const double *__restrict__ bsum,
                                                                 uint64_t n, const double *__restrict__ draws, uint32_t c, double target_in,
                                                                 double offset_in, const float *__restrict__ rows, uint32_t dim,
                                                                 float *cen, uint32_t *sel, double *total_out, long long *pick_out) {
    __shared__ double warp_tot[32];
    __shared__ unsigned long long s_blk;
    __shared__ double s_off;
    __shared__ unsigned s_row;
    const uint32_t tid = threadIdx.x;
    const uint64_t nblk = (n + KPP_BLOCK - 1) / KPP_BLOCK;
    // each thread owns a contiguous run of blocks: its sequential sum, then the CTA scan of the runs
    const uint64_t per = (nblk + SEL_THREADS - 1) / SEL_THREADS;
    const uint64_t b0 = (uint64_t)tid * per < nblk ? (uint64_t)tid * per : nblk, b1 = b0 + per < nblk ? b0 + per : nblk;
    double mine = 0.0;
    for (uint64_t b = b0; b < b1; ++b) mine += bsum[b];
    double total;
    const double excl = cta_exclusive_scan(mine, warp_tot, &total);
    if (mode == KPP_TOTAL) {
        if (tid == 0) *total_out = total;
        return;
    }
    const double target = mode == KPP_SELECT ? draws[c - 1] * total : target_in;
    const double off0 = mode == KPP_SELECT ? 0.0 : offset_in;
    if (tid == 0) s_blk = ULLONG_MAX;
    __syncthreads();
    // first block with offset + block sum >= target (cumWeight >= target, kmeans.go:400-406); NaN never compares true
    uint64_t found = ULLONG_MAX;
    double off = off0 + excl, found_off = 0.0;
    for (uint64_t b = b0; b < b1; ++b) {
        const double v = off + bsum[b];
        if (v >= target) { found = b; found_off = off; break; }
        off = v;
    }
    if (found != ULLONG_MAX) atomicMin(&s_blk, (unsigned long long)found);
    __syncthreads();
    if (found != ULLONG_MAX && found == s_blk) s_off = found_off;
    __syncthreads();
    long long pick = -1;
    uint64_t blk = s_blk;
    double boff = s_off;
    for (; blk < nblk; ++blk) {
        const uint64_t i = blk * KPP_BLOCK + tid;
        double tot;
        const double cum = cta_inclusive_scan(i < n ? d2[i] : 0.0, warp_tot, &tot);
        if (tid == 0) s_row = UINT_MAX;
        __syncthreads();
        if (i < n && boff + cum >= target) atomicMin(&s_row, tid);
        __syncthreads();
        if (s_row != UINT_MAX) { pick = (long long)(blk * KPP_BLOCK + s_row); break; }
        boff += bsum[blk];  // fell short by rounding: the next block starts at this block's running offset
    }
    if (mode == KPP_SELECT_AT) {
        if (tid == 0) *pick_out = pick;
        return;
    }
    const uint64_t r = pick < 0 ? n - 1 : (uint64_t)pick;  // selectedIdx := n - 1 (kmeans.go:398)
    if (tid == 0) sel[c] = (uint32_t)r;
    for (uint32_t k = tid; k < dim; k += SEL_THREADS) cen[(size_t)c * dim + k] = rows[r * dim + k];
}

__global__ void __launch_bounds__(256) kpp_cc_kernel(const float *__restrict__ cen, uint32_t c, uint32_t dim, bool vec4,
                                                     double *__restrict__ cc) {
    const int lane = threadIdx.x & 31;
    const uint32_t j = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (j >= c) return;  // warp-uniform
    const double s = warp_sq_euclid<false>(cen + (size_t)j * dim, cen + (size_t)c * dim, dim, vec4, lane);
    if (lane == 0) cc[j] = sqrt(s);
}

int launch_status(const char *what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return -1;
    }
    return 0;
}

}  // namespace

int kpp_update(const DeviceInfo &di, const float *rows, uint64_t n, uint32_t dim, const float *cen, uint32_t c, bool init,
               const double *cc, double *d2, int32_t *near, double *bsum, unsigned long long *scored, cudaStream_t s) {
    if (n == 0) return 0;
    static int per_sm = 0;  // same kernel and architecture on every device of the process
    if (per_sm == 0) {
        int b = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kpp_update_kernel, UPD_THREADS, 0) != cudaSuccess || b < 1) b = 1;
        per_sm = b;
    }
    const uint64_t nblk = (n + KPP_BLOCK - 1) / KPP_BLOCK;
    const unsigned grid = (unsigned)std::min<uint64_t>(nblk, (uint64_t)di.num_sms * per_sm);
    // 16-byte loads need dim % 4 == 0 and 16-byte aligned bases (caller-owned rows may start anywhere)
    const bool vec4 = dim % 4 == 0 && reinterpret_cast<uintptr_t>(rows) % 16 == 0 && reinterpret_cast<uintptr_t>(cen) % 16 == 0;
    kpp_update_kernel<<<grid, UPD_THREADS, 0, s>>>(rows, n, dim, vec4, cen, c, init, cc, d2, near, bsum, scored);
    return launch_status("kpp_update");
}

int kpp_select(int mode, const double *d2, const double *bsum, uint64_t n, const double *draws, uint32_t c, double target,
               double offset, const float *rows, uint32_t dim, float *cen, uint32_t *sel, double *total_out, long long *pick_out,
               cudaStream_t s) {
    kpp_select_kernel<<<1, SEL_THREADS, 0, s>>>(mode, d2, bsum, n, draws, c, target, offset, rows, dim, cen, sel, total_out, pick_out);
    return launch_status("kpp_select");
}

int kpp_cc(const float *cen, uint32_t c, uint32_t dim, double *cc, cudaStream_t s) {
    if (c == 0) return 0;
    const bool vec4 = dim % 4 == 0 && reinterpret_cast<uintptr_t>(cen) % 16 == 0;
    kpp_cc_kernel<<<(c + 7) / 8, 256, 0, s>>>(cen, c, dim, vec4, cc);
    return launch_status("kpp_cc");
}

}  // namespace nk
