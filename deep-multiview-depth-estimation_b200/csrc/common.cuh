// Shared host/device helpers for libmvs_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>
#include "../../include/mvs_b200.h"

namespace mvsb200 {

extern thread_local char g_err[512];
extern std::atomic<uint64_t> g_launches;

#define MVS_FAIL(code, ...)                                         \
    do {                                                            \
        snprintf(::mvsb200::g_err, sizeof(::mvsb200::g_err), __VA_ARGS__); \
        return (code);                                              \
    } while (0)

#define MVS_REQUIRE(cond, ...)                                      \
    do {                                                            \
        if (!(cond)) MVS_FAIL(MVSB200_E_BADARG, __VA_ARGS__);       \
    } while (0)

// call right after a kernel launch
#define MVS_CHECK_LAUNCH(name)                                      \
    do {                                                            \
        ::mvsb200::g_launches.fetch_add(1, std::memory_order_relaxed); \
        cudaError_t e_ = cudaGetLastError();                        \
        if (e_ != cudaSuccess)                                      \
            MVS_FAIL(MVSB200_E_LAUNCH, "%s: %s", name, cudaGetErrorString(e_)); \
    } while (0)

#define MVS_CUDA(call)                                              \
    do {                                                            \
        cudaError_t e_ = (call);                                    \
        if (e_ != cudaSuccess)                                      \
            MVS_FAIL(MVSB200_E_LAUNCH, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

// return the error of a call that reports one (MVSB200_OK = 0 otherwise)
#define MVS_TRY(call)                                               \
    do {                                                            \
        const int rc_ = (call);                                     \
        if (rc_ != MVSB200_OK) return rc_;                          \
    } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// SM count of the current device; 148 (a B200) if the query fails
inline int sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) return n;
    return 148;
}

// Unsigned 32-bit division by a run-time constant without a divide instruction (multiply-high + shift; the branch-free
// scheme of Granlund & Montgomery as used by libdivide; exact for every 32-bit numerator, checked by brute force on the host).
// The streaming kernels decode a flat chunk index into (b, d, y, x, channel group) per 16 bytes moved: with `/` and `%` on
// run-time extents that decode cost more instructions than the arithmetic on the data.
struct FastDiv {
    unsigned d, magic, shift;
};
inline FastDiv make_fastdiv(unsigned d) {
    FastDiv f;
    f.d = d; f.magic = 0; f.shift = 0;
    if (d <= 1) return f;
    const unsigned l = 31 - (unsigned)__builtin_clz(d);
    if ((d & (d - 1)) == 0) { f.shift = l - 1; return f; }
    const uint64_t num = (uint64_t)1 << (32 + l);
    uint32_t m = (uint32_t)(num / d);
    const uint32_t rem = (uint32_t)(num % d);
    m += m;
    const uint32_t twice = rem + rem;
    if (twice >= d || twice < rem) m += 1;
    f.magic = m + 1; f.shift = l;
    return f;
}
__device__ __forceinline__ unsigned fd_div(unsigned n, const FastDiv& f) {
    const unsigned q = __umulhi(n, f.magic);
    const unsigned t = ((n - q) >> 1) + q;
    return f.d == 1 ? n : (t >> f.shift);
}
// n -> (n / d, n % d)
__device__ __forceinline__ unsigned fd_divmod(unsigned n, const FastDiv& f, unsigned& rem) {
    const unsigned q = fd_div(n, f);
    rem = n - q * f.d;
    return q;
}

// streaming 16-byte store that does NOT allocate in L1: cost volumes are far larger than L2 and are read once, and an
// L1-allocating store stream evicts the feature-map lines the tap loads live on (profiles/k1 notes)
__device__ __forceinline__ void st_cs_f4(float4* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void st_cs_u4(uint4* p, uint4 v) {
    asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void st_cs_u2(void* p, uint32_t a, uint32_t b) {
    asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ float4 ld_cs_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.cs.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// one axis of torch's upsample_bilinear2d with align_corners = False (refine_input, the colours of the fused point cloud):
// src = (o + 0.5) * scale - 0.5 clamped at 0, taps i0 and i0 + step (clamped at the border), weights l0 and l1
struct Tap { int i0, step; float l0, l1; };

__device__ __forceinline__ Tap tap_of(int o, float scale, int n_in) {
    float src = scale * ((float)o + 0.5f) - 0.5f;
    src = src < 0.f ? 0.f : src;
    Tap t;
    t.i0 = min((int)src, n_in - 1);
    t.step = t.i0 < n_in - 1 ? 1 : 0;
    t.l1 = src - (float)t.i0;
    t.l0 = 1.f - t.l1;
    return t;
}

}  // namespace mvsb200
