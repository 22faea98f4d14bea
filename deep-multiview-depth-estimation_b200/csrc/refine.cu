// The glue either side of the depth-refinement network (SURVEY §8 row f2), one launch each way.
//
// Reference semantics (/root/reference/scripts/model.py:190-205):
//   norm    = (initial - d_min[b]) / span[b]                          span = d_int * D_NUM * D_SCALE
//   input   = cat(norm, bilinear resize of the reference image to the feature resolution)      [B, 4, h, w]
//   refined = (DepthRefinement(input) + norm) * span[b] + d_min[b]    (model.py:150-151: the network adds its residual to norm)
// Written with torch that is ~10 elementwise / resize / concat launches on 80 KB maps, and as many in the backward.  Here:
//   refine_input_fwd   one thread per output pixel: norm (kept in fp32 for the residual) and the 4 data channels of a bf16
//                      channel-last row of `cp` channels (the rest zeros) -- the layout the tcgen05 convolution's TMA box reads;
//   refine_input_bwd   d initial = (g_row[0] + g_norm) / span;
//   refine_output_fwd  refined = (residual + norm) * span + d_min  from channel 0 of the last convolution's rows;
//   refine_output_bwd  g_residual row (channel 0 = g * span, the rest zeros) and g_norm = g * span.
// The resize is torch's upsample_bilinear2d with align_corners = False: src = (dst + 0.5) * (in / out) - 0.5 clamped at 0,
// taps floor(src) and its successor (clamped at the border), weights 1 - frac and frac.
#include "common.cuh"
#include <cuda_bf16.h>
using namespace mvsb200;

namespace {

constexpr int kRefThreads = 128;

template <int CP>
__global__ void __launch_bounds__(kRefThreads) refine_input_fwd_kernel(
        const float* __restrict__ initial, const float* __restrict__ images, long long s_n, long long s_c, long long s_h, long long s_w,
        int n_views, int H, int W, const float* __restrict__ d_min, const float* __restrict__ span, int B, int h, int w,
        __nv_bfloat16* __restrict__ rows, float* __restrict__ norm) {
    const long long i = (long long)blockIdx.x * kRefThreads + threadIdx.x;
    if (i >= (long long)B * h * w) return;
    const int x = (int)(i % w), y = (int)((i / w) % h), b = (int)(i / ((long long)w * h));
    const float nv = (initial[i] - d_min[b]) / span[b];
    norm[i] = nv;
    const Tap ty = tap_of(y, (float)H / (float)h, H), tx = tap_of(x, (float)W / (float)w, W);
    const float* img = images + (long long)b * n_views * s_n + ty.i0 * s_h + tx.i0 * s_w;
    __align__(16) __nv_bfloat16 v[CP];
#pragma unroll
    for (int c = 0; c < CP; ++c) v[c] = __float2bfloat16(0.f);
    v[0] = __float2bfloat16(nv);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float* p = img + c * s_c;
        const float a = p[0], bq = p[tx.step * s_w], cq = p[ty.step * s_h], d = p[ty.step * s_h + tx.step * s_w];
        v[1 + c] = __float2bfloat16(ty.l0 * (tx.l0 * a + tx.l1 * bq) + ty.l1 * (tx.l0 * cq + tx.l1 * d));
    }
    uint4* dst = reinterpret_cast<uint4*>(rows + i * CP);
#pragma unroll
    for (int q = 0; q < CP / 8; ++q) dst[q] = reinterpret_cast<const uint4*>(v)[q];
}

__global__ void __launch_bounds__(kRefThreads) refine_input_bwd_kernel(const __nv_bfloat16* __restrict__ g_rows, int cp,
                                                                       const float* __restrict__ g_norm, const float* __restrict__ span,
                                                                       int B, int n, float* __restrict__ g_initial) {
    const long long i = (long long)blockIdx.x * kRefThreads + threadIdx.x;
    if (i >= (long long)B * n) return;
    float g = g_norm ? g_norm[i] : 0.f;
    if (g_rows) g += __bfloat162float(g_rows[i * cp]);
    g_initial[i] = g / span[i / n];
}

__global__ void __launch_bounds__(kRefThreads) refine_output_fwd_kernel(const __nv_bfloat16* __restrict__ res_rows, int cr,
                                                                        const float* __restrict__ norm, const float* __restrict__ d_min,
                                                                        const float* __restrict__ span, int B, int n,
                                                                        float* __restrict__ refined) {
    const long long i = (long long)blockIdx.x * kRefThreads + threadIdx.x;
    if (i >= (long long)B * n) return;
    const int b = (int)(i / n);
    refined[i] = (__bfloat162float(res_rows[i * cr]) + norm[i]) * span[b] + d_min[b];
}

template <int CR>
__global__ void __launch_bounds__(kRefThreads) refine_output_bwd_kernel(const float* __restrict__ g, const float* __restrict__ span,
                                                                        int B, int n, __nv_bfloat16* __restrict__ g_rows,
                                                                        float* __restrict__ g_norm) {
    const long long i = (long long)blockIdx.x * kRefThreads + threadIdx.x;
    if (i >= (long long)B * n) return;
    const float v = g[i] * span[i / n];
    g_norm[i] = v;
    __align__(16) __nv_bfloat16 r[CR];
#pragma unroll
    for (int c = 0; c < CR; ++c) r[c] = __float2bfloat16(0.f);
    r[0] = __float2bfloat16(v);
    uint4* dst = reinterpret_cast<uint4*>(g_rows + i * CR);
#pragma unroll
    for (int q = 0; q < CR / 8; ++q) dst[q] = reinterpret_cast<const uint4*>(r)[q];
}

inline unsigned blocks_for(long long n) { return (unsigned)((n + kRefThreads - 1) / kRefThreads); }

}  // namespace

extern "C" int mvsb200_refine_input_fwd(const float* initial, const float* images, const int64_t* image_strides4_host, int n_views,
                                        int H, int W, const float* d_min, const float* span, int B, int h, int w, int cp, void* rows,
                                        float* norm, void* stream) {
    MVS_REQUIRE(initial && images && image_strides4_host && d_min && span && rows && norm, "refine_input_fwd: null pointer");
    MVS_REQUIRE(B >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1 && n_views >= 1, "refine_input_fwd: bad shape");
    MVS_REQUIRE(cp == 8 || cp == 16, "refine_input_fwd: rows of 8 or 16 channels (got %d)", cp);
    const long long tot = (long long)B * h * w;
    const int64_t* s = image_strides4_host;
    if (cp == 8)
        refine_input_fwd_kernel<8><<<blocks_for(tot), kRefThreads, 0, (cudaStream_t)stream>>>(
            initial, images, s[0], s[1], s[2], s[3], n_views, H, W, d_min, span, B, h, w, (__nv_bfloat16*)rows, norm);
    else
        refine_input_fwd_kernel<16><<<blocks_for(tot), kRefThreads, 0, (cudaStream_t)stream>>>(
            initial, images, s[0], s[1], s[2], s[3], n_views, H, W, d_min, span, B, h, w, (__nv_bfloat16*)rows, norm);
    MVS_CHECK_LAUNCH("refine_input_fwd");
    return MVSB200_OK;
}

extern "C" int mvsb200_refine_input_bwd(const void* g_rows, int cp, const float* g_norm, const float* span, int B, int n,
                                        float* g_initial, void* stream) {
    MVS_REQUIRE((g_rows || g_norm) && span && g_initial, "refine_input_bwd: null pointer");
    MVS_REQUIRE(B >= 1 && n >= 1 && cp >= 1, "refine_input_bwd: bad shape");
    refine_input_bwd_kernel<<<blocks_for((long long)B * n), kRefThreads, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)g_rows, cp, g_norm, span, B, n, g_initial);
    MVS_CHECK_LAUNCH("refine_input_bwd");
    return MVSB200_OK;
}

extern "C" int mvsb200_refine_output_fwd(const void* res_rows, int cr, const float* norm, const float* d_min, const float* span,
                                         int B, int n, float* refined, void* stream) {
    MVS_REQUIRE(res_rows && norm && d_min && span && refined, "refine_output_fwd: null pointer");
    MVS_REQUIRE(B >= 1 && n >= 1 && cr >= 1, "refine_output_fwd: bad shape");
    refine_output_fwd_kernel<<<blocks_for((long long)B * n), kRefThreads, 0, (cudaStream_t)stream>>>(
        (const __nv_bfloat16*)res_rows, cr, norm, d_min, span, B, n, refined);
    MVS_CHECK_LAUNCH("refine_output_fwd");
    return MVSB200_OK;
}

extern "C" int mvsb200_refine_output_bwd(const float* g_refined, const float* span, int B, int n, int cr, void* g_rows, float* g_norm,
                                         void* stream) {
    MVS_REQUIRE(g_refined && span && g_rows && g_norm, "refine_output_bwd: null pointer");
    MVS_REQUIRE(B >= 1 && n >= 1, "refine_output_bwd: bad shape");
    MVS_REQUIRE(cr == 8 || cr == 16, "refine_output_bwd: rows of 8 or 16 channels (got %d)", cr);
    if (cr == 8)
        refine_output_bwd_kernel<8><<<blocks_for((long long)B * n), kRefThreads, 0, (cudaStream_t)stream>>>(
            g_refined, span, B, n, (__nv_bfloat16*)g_rows, g_norm);
    else
        refine_output_bwd_kernel<16><<<blocks_for((long long)B * n), kRefThreads, 0, (cudaStream_t)stream>>>(
            g_refined, span, B, n, (__nv_bfloat16*)g_rows, g_norm);
    MVS_CHECK_LAUNCH("refine_output_bwd");
    return MVSB200_OK;
}
