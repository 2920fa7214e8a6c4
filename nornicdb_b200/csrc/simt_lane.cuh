// simt_lane.cuh — the CUDA-core scan's per-lane pieces, shared by the full scan (scan_simt.cu) and the cluster-routed
// scan (cluster_search.cu): 16-byte row loaders and the butterfly reduce-scatter.  Both kernels accumulate a (row, query)
// score with the same per-lane order and the same reduction tree, so they return bit-identical scores for the same row.
#pragma once
#include "kernels.cuh"

namespace nk {

// ---- element loaders -------------------------------------------------------------------------
template <typename T, bool VEC> struct Lane;
template <> struct Lane<float, true> {
    static constexpr int EPL = 4;
    static __device__ __forceinline__ void load(const float *p, float (&x)[4]) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(x[0]), "=f"(x[1]), "=f"(x[2]), "=f"(x[3]) : "l"(p));
    }
};
template <> struct Lane<__half, true> {
    static constexpr int EPL = 8;
    static __device__ __forceinline__ void load(const __half *p, float (&x)[8]) {
        uint32_t w0, w1, w2, w3;
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "l"(p));
        float2 f;
        f = __half22float2(*reinterpret_cast<__half2 *>(&w0)); x[0] = f.x; x[1] = f.y;
        f = __half22float2(*reinterpret_cast<__half2 *>(&w1)); x[2] = f.x; x[3] = f.y;
        f = __half22float2(*reinterpret_cast<__half2 *>(&w2)); x[4] = f.x; x[5] = f.y;
        f = __half22float2(*reinterpret_cast<__half2 *>(&w3)); x[6] = f.x; x[7] = f.y;
    }
};
template <> struct Lane<__nv_bfloat16, true> {
    static constexpr int EPL = 8;
    static __device__ __forceinline__ void load(const __nv_bfloat16 *p, float (&x)[8]) {
        uint32_t w[4];
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "l"(p));
#pragma unroll
        for (int i = 0; i < 4; ++i) {  // bf16 -> fp32 is a 16-bit shift
            x[2 * i] = __uint_as_float(w[i] << 16);
            x[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
};
template <> struct Lane<__nv_bfloat16, false> {
    static constexpr int EPL = 1;
    static __device__ __forceinline__ void load(const __nv_bfloat16 *p, float (&x)[1]) { x[0] = __bfloat162float(*p); }
};
template <> struct Lane<float, false> {
    static constexpr int EPL = 1;
    static __device__ __forceinline__ void load(const float *p, float (&x)[1]) { x[0] = __ldg(p); }
};
template <> struct Lane<__half, false> {
    static constexpr int EPL = 1;
    static __device__ __forceinline__ void load(const __half *p, float (&x)[1]) { x[0] = __half2float(__ldg(p)); }
};

// Butterfly reduce-scatter of V per-lane partial sums across the warp.  Afterwards v[0] holds the
// finished total of value index lane / (32 / V) (every lane of that group holds the same total).
template <int V>
__device__ __forceinline__ void warp_reduce_scatter(float (&v)[V], int lane) {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const int o = 16 >> s;
        const int c = V >> s;  // live values before this step (compile-time after unrolling)
        if (c > 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < (c >> 1); ++i) {
                float keep = up ? v[i + (c >> 1)] : v[i];
                float send = up ? v[i] : v[i + (c >> 1)];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
            }
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
        }
    }
}

}  // namespace nk
