// K4: depth-axis softmax + the reference's "top-N" expected depth, forward and backward (sm_100a).
//
// Reference semantics (citations into /root/reference/scripts):
//   model.py:96,123     prob = Softmax(dim=2)(conv_out(...))               [B,1,D,h,w]
//   depthmap.py:11-19   idx = argsort_desc_D(prob); mask[k] = idx[k] < N_DEPTH_EST; the mask is applied
//                       POSITIONALLY to the unsorted volume, so the planes kept are {rank(j) : j < N}
//                       where rank(j) is the position of plane j in the descending sort (SURVEY App. A.6);
//                       depth = sum_kept d[k] P[k] / sum_kept P[k].
// No sort is needed: rank(j) = #{k : P[k] > P[j]} + #{k < j : P[k] == P[j]}  (stable descending).
//
// Layout: [B, D, h, w] fp32, the D values of a pixel are h*w apart => lanes run along x (coalesced
// 128 B rows per plane), a CTA stages a [D][32 pixel] tile in shared memory so HBM is read exactly
// once, and the D-axis reductions run across the CTA's 8 warps + shared memory.
#include "common.cuh"

using namespace mvsb200;

namespace {

constexpr int kPix = 32;       // pixels per CTA (one warp-width of x)
constexpr int kSlices = 8;     // warps per CTA, each owning planes d = slice (mod 8)
constexpr int kMaxKeep = 8;

// MVSNet's photometric confidence: the probability mass of the (up to) four planes around the estimate.  t = (depth - d_0) /
// (d_1 - d_0), k0 = floor(t); conf = sum of P[k] over k in {k0-1 .. k0+2} and [0, D-1], added in ascending k in fp32.  D == 1
// gives 1; a non-finite depth, index or summed probability gives NaN.  `p(k)` reads plane k of this pixel.
template <class ProbAt>
__device__ __forceinline__ float confidence_of(float dep, const float* __restrict__ dv, int D, ProbAt p) {
    if (!isfinite(dep)) return __int_as_float(0x7fc00000);
    if (D == 1) return 1.f;
    const float t = (dep - dv[0]) / (dv[1] - dv[0]);
    if (!isfinite(t)) return __int_as_float(0x7fc00000);
    const float k0f = floorf(t);
    if (k0f < -3.f || k0f > (float)D + 1.f) return 0.f;      // the window misses [0, D-1]
    const int k0 = (int)k0f;
    float s = 0.f;
    for (int k = max(k0 - 1, 0); k <= min(k0 + 2, D - 1); ++k) s += p(k);
    return isfinite(s) ? s : __int_as_float(0x7fc00000);
}

// CONF: also write the confidence of every pixel (conf != nullptr, depth required); the plain form keeps its code unchanged
template <bool CONF>
__global__ void __launch_bounds__(kPix * kSlices) softmax_depth_fwd_kernel(const float* __restrict__ in, int apply_softmax,
                                                                        const float* __restrict__ depths,
                                                                        float* __restrict__ prob, int32_t* __restrict__ ranks,
                                                                        float* __restrict__ depth, float* __restrict__ conf,
                                                                        int D, int hw, int n_keep) {
    extern __shared__ float smem[];
    float* tile = smem;                          // [D][kPix]
    float* red = smem + (size_t)D * kPix;        // [kSlices][kPix]
    int* cnt = reinterpret_cast<int*>(red + kSlices * kPix);   // [kMaxKeep][kPix]
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int b = blockIdx.y;
    const int pix = blockIdx.x * kPix + lane;
    const bool ok = pix < hw;
    const float* src = in + (size_t)b * D * hw + pix;

    float mx = -INFINITY;
    for (int d = slice; d < D; d += kSlices) {
        const float v = ok ? __ldcs(src + (size_t)d * hw) : 0.f;
        tile[d * kPix + lane] = v;
        mx = fmaxf(mx, v);
    }
    if (threadIdx.x < kMaxKeep * kPix) cnt[threadIdx.x] = 0;
    if (apply_softmax) {
        red[slice * kPix + lane] = mx;
        __syncthreads();
        mx = red[lane];
#pragma unroll
        for (int s = 1; s < kSlices; ++s) mx = fmaxf(mx, red[s * kPix + lane]);
        __syncthreads();
        float sum = 0.f;
        for (int d = slice; d < D; d += kSlices) {
            const float e = expf(tile[d * kPix + lane] - mx);
            tile[d * kPix + lane] = e;
            sum += e;
        }
        red[slice * kPix + lane] = sum;
        __syncthreads();
        sum = red[lane];
#pragma unroll
        for (int s = 1; s < kSlices; ++s) sum += red[s * kPix + lane];
        float* dst = prob + (size_t)b * D * hw + pix;
        for (int d = slice; d < D; d += kSlices) {
            const float p = tile[d * kPix + lane] / sum;     // torch: exp(x - max) / sum
            tile[d * kPix + lane] = p;
            if (ok) dst[(size_t)d * hw] = p;
        }
    }
    __syncthreads();
    if (!ranks && !depth) return;

    // stable descending rank of planes 0..n_keep-1
    float pj[kMaxKeep];
    int c[kMaxKeep];
#pragma unroll
    for (int j = 0; j < kMaxKeep; ++j) {
        pj[j] = j < n_keep ? tile[j * kPix + lane] : 0.f;
        c[j] = 0;
    }
    for (int d = slice; d < D; d += kSlices) {
        const float p = tile[d * kPix + lane];
#pragma unroll
        for (int j = 0; j < kMaxKeep; ++j) c[j] += (p > pj[j]) || (p == pj[j] && d < j);
    }
#pragma unroll
    for (int j = 0; j < kMaxKeep; ++j)
        if (j < n_keep) atomicAdd(&cnt[j * kPix + lane], c[j]);
    __syncthreads();
    if (slice == 0 && ok) {
        float num = 0.f, den = 0.f;
        for (int j = 0; j < n_keep; ++j) {
            const int r = cnt[j * kPix + lane];
            if (ranks) ranks[((size_t)b * n_keep + j) * hw + pix] = r;
            if (depth) {
                const float p = tile[r * kPix + lane];
                num = fmaf(depths[(size_t)b * D + r], p, num);
                den += p;
            }
        }
        if (depth) depth[(size_t)b * hw + pix] = num / den;
        if constexpr (CONF)
            conf[(size_t)b * hw + pix] = confidence_of(num / den, depths + (size_t)b * D, D, [&](int k) { return tile[k * kPix + lane]; });
    }
}

__global__ void depth_confidence_kernel(const float* __restrict__ prob, const float* __restrict__ depth, const float* __restrict__ depths,
                                        float* __restrict__ conf, int D, int hw) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (pix >= hw) return;
    const float* col = prob + (size_t)b * D * hw + pix;
    conf[(size_t)b * hw + pix] = confidence_of(depth[(size_t)b * hw + pix], depths + (size_t)b * D, D,
                                               [&](int k) { return col[(size_t)k * hw]; });
}

__global__ void depth_from_ranks_kernel(const float* __restrict__ prob, const int32_t* __restrict__ ranks,
                                        const float* __restrict__ depths, float* __restrict__ depth, int D, int hw, int n_keep) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (pix >= hw) return;
    float num = 0.f, den = 0.f;
    for (int j = 0; j < n_keep; ++j) {
        const int r = ranks[((size_t)b * n_keep + j) * hw + pix];
        const float p = prob[((size_t)b * D + r) * hw + pix];
        num = fmaf(depths[(size_t)b * D + r], p, num);
        den += p;
    }
    depth[(size_t)b * hw + pix] = num / den;
}

// gprob[b,k,pix] = gdepth * (d_k - depth) / S for the kept planes, 0 elsewhere
__global__ void depth_bwd_kernel(const float* __restrict__ prob, const int32_t* __restrict__ ranks,
                                 const float* __restrict__ depths, const float* __restrict__ gdepth,
                                 float* __restrict__ gprob, int D, int hw, int n_keep) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
    if (pix >= hw) return;
    int r[kMaxKeep];
    float num = 0.f, den = 0.f;
#pragma unroll
    for (int j = 0; j < kMaxKeep; ++j) {
        r[j] = -1;
        if (j < n_keep) {
            r[j] = ranks[((size_t)b * n_keep + j) * hw + pix];
            const float p = prob[((size_t)b * D + r[j]) * hw + pix];
            num = fmaf(depths[(size_t)b * D + r[j]], p, num);
            den += p;
        }
    }
    const float dep = num / den, gs = gdepth[(size_t)b * hw + pix] / den;
    float* dst = gprob + (size_t)b * D * hw + pix;
    for (int d = 0; d < D; ++d) {
        bool kept = false;
#pragma unroll
        for (int j = 0; j < kMaxKeep; ++j) kept |= (r[j] == d);
        dst[(size_t)d * hw] = kept ? gs * (depths[(size_t)b * D + d] - dep) : 0.f;
    }
}

// glogits = P * (g - sum_D g P)
__global__ void __launch_bounds__(kPix * kSlices) softmax_bwd_kernel(const float* __restrict__ prob, const float* __restrict__ gprob,
                                                                  float* __restrict__ glogits, int D, int hw) {
    __shared__ float red[kSlices][kPix];
    const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int b = blockIdx.y, pix = blockIdx.x * kPix + lane;
    const bool ok = pix < hw;
    const size_t base = (size_t)b * D * hw + pix;
    float dot = 0.f;
    for (int d = slice; d < D; d += kSlices)
        if (ok) dot = fmaf(prob[base + (size_t)d * hw], gprob[base + (size_t)d * hw], dot);
    red[slice][lane] = dot;
    __syncthreads();
    dot = 0.f;
#pragma unroll
    for (int s = 0; s < kSlices; ++s) dot += red[s][lane];
    for (int d = slice; d < D; d += kSlices)
        if (ok) glogits[base + (size_t)d * hw] = prob[base + (size_t)d * hw] * (gprob[base + (size_t)d * hw] - dot);
}

}  // namespace

template <bool CONF>
static int softmax_depth_launch(const char* name, const float* in, int apply_softmax, const float* depths, float* prob,
                                int32_t* ranks, float* depth, float* conf, int B, int D, int h, int w, int n_est, void* stream) {
    MVS_REQUIRE(in, "%s: null input", name);
    MVS_REQUIRE(!apply_softmax || prob, "%s: prob output required with apply_softmax", name);
    MVS_REQUIRE((depth != nullptr) == (depths != nullptr), "%s: depth and depths go together", name);
    MVS_REQUIRE(!CONF || (conf && depth), "%s: conf and depth outputs required", name);
    MVS_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && D <= 1024 && h >= 1 && w >= 1, "%s: bad shape", name);
    MVS_REQUIRE(n_est >= 1 && n_est <= kMaxKeep, "%s: 1 <= n_est <= %d", name, kMaxKeep);
    const int hw = h * w, n_keep = n_est < D ? n_est : D;
    const size_t smem = ((size_t)D * kPix + kSlices * kPix) * sizeof(float) + kMaxKeep * kPix * sizeof(int);
    if (smem > 48 * 1024)   // per-device attribute; cheap, so set whenever the opt-in range is needed
        MVS_CUDA(cudaFuncSetAttribute(softmax_depth_fwd_kernel<CONF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    dim3 grid((hw + kPix - 1) / kPix, B);
    softmax_depth_fwd_kernel<CONF><<<grid, kPix * kSlices, smem, (cudaStream_t)stream>>>(in, apply_softmax, depths, prob, ranks,
                                                                                        depth, conf, D, hw, n_keep);
    MVS_CHECK_LAUNCH(name);
    return MVSB200_OK;
}

extern "C" int mvsb200_softmax_depth_fwd(const float* in, int apply_softmax, const float* depths, float* prob,
                                         int32_t* ranks, float* depth, int B, int D, int h, int w, int n_est, void* stream) {
    return softmax_depth_launch<false>("softmax_depth_fwd", in, apply_softmax, depths, prob, ranks, depth, nullptr, B, D, h, w,
                                       n_est, stream);
}

extern "C" int mvsb200_softmax_depth_conf_fwd(const float* in, int apply_softmax, const float* depths, float* prob,
                                              int32_t* ranks, float* depth, float* conf, int B, int D, int h, int w, int n_est,
                                              void* stream) {
    return softmax_depth_launch<true>("softmax_depth_conf_fwd", in, apply_softmax, depths, prob, ranks, depth, conf, B, D, h, w,
                                      n_est, stream);
}

extern "C" int mvsb200_depth_confidence(const float* prob, const float* depth, const float* depths, float* conf, int B, int D,
                                        int h, int w, void* stream) {
    MVS_REQUIRE(prob && depth && depths && conf, "depth_confidence: null pointer");
    MVS_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && h >= 1 && w >= 1, "depth_confidence: bad shape");
    const int hw = h * w;
    dim3 grid((hw + 127) / 128, B);
    depth_confidence_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(prob, depth, depths, conf, D, hw);
    MVS_CHECK_LAUNCH("depth_confidence");
    return MVSB200_OK;
}

extern "C" int mvsb200_depth_from_ranks(const float* prob, const int32_t* ranks, const float* depths, float* depth, int B,
                                        int D, int h, int w, int n_keep, void* stream) {
    MVS_REQUIRE(prob && ranks && depths && depth, "depth_from_ranks: null pointer");
    MVS_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && n_keep >= 1 && n_keep <= kMaxKeep && n_keep <= D, "depth_from_ranks: bad shape");
    const int hw = h * w;
    dim3 grid((hw + 127) / 128, B);
    depth_from_ranks_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(prob, ranks, depths, depth, D, hw, n_keep);
    MVS_CHECK_LAUNCH("depth_from_ranks");
    return MVSB200_OK;
}

extern "C" int mvsb200_depth_bwd(const float* prob, const int32_t* ranks, const float* depths, const float* gdepth,
                                 float* gprob, int B, int D, int h, int w, int n_keep, void* stream) {
    MVS_REQUIRE(prob && ranks && depths && gdepth && gprob, "depth_bwd: null pointer");
    MVS_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && n_keep >= 1 && n_keep <= kMaxKeep && n_keep <= D, "depth_bwd: bad shape");
    const int hw = h * w;
    dim3 grid((hw + 127) / 128, B);
    depth_bwd_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(prob, ranks, depths, gdepth, gprob, D, hw, n_keep);
    MVS_CHECK_LAUNCH("depth_bwd");
    return MVSB200_OK;
}

extern "C" int mvsb200_softmax_bwd(const float* prob, const float* gprob, float* glogits, int B, int D, int h, int w,
                                   void* stream) {
    MVS_REQUIRE(prob && gprob && glogits, "softmax_bwd: null pointer");
    MVS_REQUIRE(B >= 1 && B <= 65535 && D >= 1 && h >= 1 && w >= 1, "softmax_bwd: bad shape");
    const int hw = h * w;
    dim3 grid((hw + kPix - 1) / kPix, B);
    softmax_bwd_kernel<<<grid, kPix * kSlices, 0, (cudaStream_t)stream>>>(prob, gprob, glogits, D, hw);
    MVS_CHECK_LAUNCH("softmax_bwd");
    return MVSB200_OK;
}
