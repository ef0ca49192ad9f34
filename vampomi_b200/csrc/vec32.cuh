// Shared device helpers of the matrix kernels: the 32-byte streaming vector (4 x FP64 or 8 x FP32 per LDG.E.256), the
// small-vector loader, 256-bit stores and the warp reduction.
#pragma once
#include <cuda_runtime.h>

namespace vampomi {

struct __align__(32) d4 { double x, y, z, w; };

// One 32-byte piece of a column of A, widened to FP64: 4 markers' values in FP64 storage, 8 in FP32 storage (opt-in,
// vampomi_create_ex). Every thread keeps the same number of BYTES in flight in both modes; arithmetic is FP64 in both.
//   stream(): LDG.E.256 on the read-only path without L1 allocation (A is touched once per pass)
//   cached(): same but allocating in L1 (statistics read every column twice)
template <typename T> struct V32;
template <> struct V32<double> {
    static constexpr int VE = 4;
    double v[4];
    __device__ __forceinline__ double val(int e) const { return v[e]; }
    // H: L2 hint of the streaming load — 0 none, 1 L2::256B prefetch, 2 L2::evict_first, 3 both
    template <int H = 0>
    static __device__ __forceinline__ V32 stream(const double* p) {
        V32 r;
        if (H == 1)
            asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
        else if (H == 2)
            asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
        else if (H == 3)
            asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.L2::256B.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
        else
            asm volatile("ld.global.nc.L1::no_allocate.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
        return r;
    }
    static __device__ __forceinline__ V32 cached(const double* p) {
        V32 r;
        asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(r.v[0]), "=d"(r.v[1]), "=d"(r.v[2]), "=d"(r.v[3]) : "l"(p));
        return r;
    }
};
template <> struct V32<float> {      // keeps the raw FP32 values (8 registers) and widens on use, so loads in flight stay cheap
    static constexpr int VE = 8;
    float f[8];
    __device__ __forceinline__ double val(int e) const { return (double)f[e]; }
    template <int H = 0>
    static __device__ __forceinline__ V32 stream(const float* p) {
        V32 r;
        if (H == 1)
            asm volatile("ld.global.nc.L1::no_allocate.L2::256B.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=f"(r.f[0]), "=f"(r.f[1]), "=f"(r.f[2]), "=f"(r.f[3]), "=f"(r.f[4]), "=f"(r.f[5]), "=f"(r.f[6]), "=f"(r.f[7]) : "l"(p));
        else if (H == 2)
            asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=f"(r.f[0]), "=f"(r.f[1]), "=f"(r.f[2]), "=f"(r.f[3]), "=f"(r.f[4]), "=f"(r.f[5]), "=f"(r.f[6]), "=f"(r.f[7]) : "l"(p));
        else if (H == 3)
            asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.L2::256B.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=f"(r.f[0]), "=f"(r.f[1]), "=f"(r.f[2]), "=f"(r.f[3]), "=f"(r.f[4]), "=f"(r.f[5]), "=f"(r.f[6]), "=f"(r.f[7]) : "l"(p));
        else
            asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                         : "=f"(r.f[0]), "=f"(r.f[1]), "=f"(r.f[2]), "=f"(r.f[3]), "=f"(r.f[4]), "=f"(r.f[5]), "=f"(r.f[6]), "=f"(r.f[7]) : "l"(p));
        return r;
    }
    static __device__ __forceinline__ V32 cached(const float* p) {
        V32 r;
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(r.f[0]), "=f"(r.f[1]), "=f"(r.f[2]), "=f"(r.f[3]), "=f"(r.f[4]), "=f"(r.f[5]), "=f"(r.f[6]), "=f"(r.f[7]) : "l"(p));
        return r;
    }
};
// VE consecutive doubles of a small, reused N-vector (p in A^T p, w in the loo sums): L1-allocating 256-bit loads.
template <int VE> struct PV {
    double v[VE];
    static __device__ __forceinline__ PV load(const double* p) {
        PV r;
#pragma unroll
        for (int q = 0; q < VE / 4; q++)
            asm volatile("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];"
                         : "=d"(r.v[4 * q]), "=d"(r.v[4 * q + 1]), "=d"(r.v[4 * q + 2]), "=d"(r.v[4 * q + 3]) : "l"(p + 4 * q));
        return r;
    }
};
__device__ __forceinline__ void st256(double* p, const d4& v) {
    asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" :: "l"(p), "d"(v.x), "d"(v.y), "d"(v.z), "d"(v.w) : "memory");
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// smallest and largest value over the warp (fmin/fmax: a NaN loses to any number)
__device__ __forceinline__ void warp_min_max(double& lo, double& hi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
}


}  // namespace vampomi
