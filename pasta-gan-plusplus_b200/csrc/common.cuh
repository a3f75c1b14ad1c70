// Shared host/device helpers for libpgpp_sm100a.so (no torch, no pybind).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cuda_fp8.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/pgpp.h"

namespace pgpp {

void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

inline void count_launch(int n = 1) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// Ablation switches (PGPP_* environment variables, DESIGN.md section 5): read once per process, not per launch;
// pgpp_refresh_env() re-reads them (timing tools that flip a switch between launches call it).
struct EnvFlags {
    bool igemm_no_reuse, igemm_no_slab2, igemm_no_resident, igemm_no_stack, igemm_no_lean_epilogue, igemm_no_tma_store, igemm_slab9;
    bool wgrad_no_reuse, wgrad_no_pair, ba_nostream, fir_packed_no_tile;
    int igemm_debug;
};
const EnvFlags& env_flags();

#define PGPP_REQUIRE(cond, ...)                                  \
    do { if (!(cond)) { ::pgpp::set_error(__VA_ARGS__); return PGPP_ERR_INVALID; } } while (0)

#define PGPP_CUDA_OK(expr)                                                                   \
    do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) {                                    \
        ::pgpp::set_error("%s failed: %s", #expr, cudaGetErrorString(e_)); return PGPP_ERR_CUDA; } } while (0)

inline int sm_count() {
    static int cached[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// resident CTAs per SM of a kernel (cached): persistent grids are sized to exactly one full wave
template <class K>
inline int occupancy_of(K kernel, int threads, size_t smem) {
    struct Entry { const void* fn; int threads; size_t smem; int occ; };
    static thread_local Entry cache[64];
    static thread_local int used = 0;
    const void* fn = (const void*)kernel;
    for (int i = 0; i < used; i++)
        if (cache[i].fn == fn && cache[i].threads == threads && cache[i].smem == smem) return cache[i].occ;
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem) != cudaSuccess || occ < 1) occ = 1;
    if (used < 64) cache[used++] = Entry{fn, threads, smem, occ};
    return occ;
}

// scalar <-> storage conversions; math runs in float (double for f64), like the reference's
// InternalType (bias_act.cu:15-18, upfirdn2d.cu:15-18)
template <class T> struct Acc { typedef float type; };
template <> struct Acc<double> { typedef double type; };

template <class T> __device__ __forceinline__ typename Acc<T>::type to_acc(T v) { return (typename Acc<T>::type)v; }
template <> __device__ __forceinline__ float to_acc<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_acc<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }

template <class T> __device__ __forceinline__ T from_acc(typename Acc<T>::type v) { return (T)v; }
template <> __device__ __forceinline__ __half from_acc<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_acc<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// tile index -> coordinates in 32-bit arithmetic (callers guarantee fewer than 2^31 tiles): r = t % d, t /= d.  A 64-bit division by a
// runtime divisor costs ~100 instructions per thread, several times per tile in a persistent kernel.
__device__ __forceinline__ int divmod_u32(unsigned& t, unsigned d) { const unsigned q = t / d, r = t - q * d; t = q; return (int)r; }

// packed float32x2 arithmetic (sm_100a FFMA2 / FADD2): halves the instruction count of the bandwidth-bound kernels that work on the
// bf16 operand format, where the conversions and sums per byte are what limits them
typedef unsigned long long f32x2;       // two packed float32 (low word = even channel)

__device__ __forceinline__ f32x2 pack2(float lo, float hi) { return (f32x2)__float_as_uint(lo) | ((f32x2)__float_as_uint(hi) << 32); }
__device__ __forceinline__ void ffma2(f32x2& d, const f32x2 a, const f32x2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b)); }
__device__ __forceinline__ f32x2 fadd2(const f32x2 a, const f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// bf16 pair (one 32-bit word, low half = even channel) -> packed float32 pair
__device__ __forceinline__ f32x2 bf2_to_f32x2(uint32_t w) { return (f32x2)(w << 16) | ((f32x2)(w & 0xffff0000u) << 32); }

// e4m3 operand format (the opt-in fp8 inference precision): round to nearest even, satfinite (|x| > 448 -> +-448, NaN stays NaN),
// i.e. cvt.rn.satfinite.e4m3x2.f32.  Four values -> one 32-bit word, byte k = value k (channels ascending in memory).
__device__ __forceinline__ uint32_t e4m3x4(float a, float b, float c, float d) {
    const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
    const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
    return lo | (hi << 16);
}
// byte pair (low byte = even channel) -> two floats (exact: every e4m3 value is a half)
__device__ __forceinline__ float2 e4m3x2_to_float2(uint32_t pair) {
    const __half2_raw h = __nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(pair & 0xffffu), __NV_E4M3);
    return __half22float2(*reinterpret_cast<const __half2*>(&h));
}

} // namespace pgpp
