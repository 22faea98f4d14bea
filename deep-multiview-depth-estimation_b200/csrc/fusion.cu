// K7: multi-view consistency filter and point-cloud fusion (MVSNet, Yao et al. 2018, §4.2), after per-view inference.
//
// Geometry (DESIGN §4 "K7 confidence and fusion"): the depth d at pixel p = (x, y, 1) of view i is the world point
//   X = C_i + d / (n_i^T r) r,   r = R_i^T K_i^-1 p,
// and the depth of a world point in view j is n_j^T (X - C_j).  n is a per-view input: R[:, 2] for the network's sweep depths
// (the plane normal of geometry.py), R[2, :] for z-depth.  The camera table holds everything in fp32, computed in fp64 on the host.
//
//   fusion_check_kernel   one thread per reference pixel, grid row = reference view: the photometric test, then every source
//                         in table order (project, bilinear depth sample, unproject there, project back), the consistent count
//                         and fused depth; also the number of kept pixels of its block (one __syncthreads_count)
//     <VIS = true>        visibility fusion: one launch per reference view `ref`, in the caller's view order.  A pixel already
//                         marked in used[ref] is no reference (mask 0, count 0, fused = d, as an invalid pixel); a kept pixel
//                         marks, in every consistent source j, the pixel nearest its projection there: used[j, round(v), round(u)]
//   fusion_emit_kernel    same grid: the block's offset (exclusive scan of the block counts, computed on the host side with
//                         torch.cumsum) plus the rank of the pixel among the kept pixels of the block (ballots) -> xyz, rgb.
//                         View-major, row-major output; no atomics, so two runs write the same point cloud bit for bit.
//   resize_rgb_kernel     the reference images at depth resolution, the resize refine_input applies.
#include "common.cuh"

using namespace mvsb200;

namespace {

constexpr int kCam = MVSB200_FUSION_CAM_FLOATS;
constexpr int kBlk = MVSB200_FUSION_BLOCK_PIXELS;
constexpr int kMaxSrc = MVSB200_FUSION_MAX_SOURCES;
// camera table fields
constexpr int kP = 0, kM = 12, kC = 21, kN = 24;

struct F3 { float x, y, z; };

__device__ __forceinline__ F3 unproject(const float* c, float x, float y, float d) {
    const F3 r = {c[kM + 0] * x + c[kM + 1] * y + c[kM + 2], c[kM + 3] * x + c[kM + 4] * y + c[kM + 5],
                  c[kM + 6] * x + c[kM + 7] * y + c[kM + 8]};
    const float s = d * __frcp_rn(c[kN] * r.x + c[kN + 1] * r.y + c[kN + 2] * r.z);
    return {c[kC] + s * r.x, c[kC + 1] + s * r.y, c[kC + 2] + s * r.z};
}

// -> (u, v) and z of K [R | T] X
__device__ __forceinline__ float project(const float* c, F3 X, float& u, float& v) {
    const float a = c[kP + 0] * X.x + c[kP + 1] * X.y + c[kP + 2] * X.z + c[kP + 3];
    const float b = c[kP + 4] * X.x + c[kP + 5] * X.y + c[kP + 6] * X.z + c[kP + 7];
    const float z = c[kP + 8] * X.x + c[kP + 9] * X.y + c[kP + 10] * X.z + c[kP + 11];
    const float rz = __frcp_rn(z);
    u = a * rz;
    v = b * rz;
    return z;
}

__device__ __forceinline__ float depth_in(const float* c, F3 X) {
    return c[kN] * (X.x - c[kC]) + c[kN + 1] * (X.y - c[kC + 1]) + c[kN + 2] * (X.z - c[kC + 2]);
}

__device__ __forceinline__ bool usable(float d) { return isfinite(d) && d > 0.f; }

template <bool VIS>
__global__ void __launch_bounds__(kBlk) fusion_check_kernel(const float* __restrict__ depth, const float* __restrict__ conf,
                                                           const float* __restrict__ cams, const int32_t* __restrict__ sources,
                                                           int S, int h, int w, float conf_min, float reproj_px, float rel_depth,
                                                           int min_views, uint8_t* __restrict__ mask, int32_t* __restrict__ count,
                                                           float* __restrict__ fused, int32_t* __restrict__ block_counts,
                                                           int vis_ref, uint8_t* __restrict__ used) {
    __shared__ float cam_s[(1 + kMaxSrc) * kCam];   // [0]: the reference view, [1 + s]: source s
    __shared__ int src_s[kMaxSrc];
    // VIS: per source, the index of the source pixel nearest to where the test projected this thread's pixel.  Staged here from
    // the same fp32 (u, v) the test used, so the mark can never disagree with the decision (a recomputed projection could be
    // contracted differently by the compiler).
    __shared__ int mark_s[VIS ? kMaxSrc * kBlk : 1];
    const int ref = VIS ? vis_ref : (int)blockIdx.y, hw = h * w, pix = blockIdx.x * kBlk + threadIdx.x;
    if (threadIdx.x < S) src_s[threadIdx.x] = sources[(size_t)ref * S + threadIdx.x];
    __syncthreads();
    for (int i = threadIdx.x; i < (1 + S) * kCam; i += kBlk) {
        const int v = i / kCam, view = v == 0 ? ref : src_s[v - 1];
        cam_s[i] = view >= 0 ? cams[(size_t)view * kCam + i % kCam] : 0.f;
    }
    __syncthreads();

    bool keep = false;
    if (pix < hw) {
        const size_t at = (size_t)ref * hw + pix;
        const float d = depth[at];
        const float fx = (float)(pix % w), fy = (float)(pix / w);
        bool valid = conf[at] >= conf_min && usable(d);           // a NaN confidence fails the comparison
        if constexpr (VIS) valid = valid && !used[at];           // another view's point has absorbed this pixel
        int cnt = 0;
        unsigned consistent = 0;                                 // VIS: bit s = source s was consistent
        float sum = d;
        if (valid) {
            const F3 X = unproject(cam_s, fx, fy, d);
            for (int s = 0; s < S; ++s) {
                const int j = src_s[s];
                if (j < 0) continue;
                const float* cs = cam_s + (1 + s) * kCam;
                float u, v;
                const float z = project(cs, X, u, v);
                if (!(z > 0.f && u >= 0.f && u <= (float)(w - 1) && v >= 0.f && v <= (float)(h - 1))) continue;
                const int x0 = (int)floorf(u), y0 = (int)floorf(v);
                const int x1 = min(x0 + 1, w - 1), y1 = min(y0 + 1, h - 1);
                const float* dm = depth + (size_t)j * hw;
                const float d00 = __ldg(dm + y0 * w + x0), d01 = __ldg(dm + y0 * w + x1);
                const float d10 = __ldg(dm + y1 * w + x0), d11 = __ldg(dm + y1 * w + x1);
                if (!(usable(d00) && usable(d01) && usable(d10) && usable(d11))) continue;
                const float ax = u - (float)x0, ay = v - (float)y0;
                const float ds = (1.f - ay) * ((1.f - ax) * d00 + ax * d01) + ay * ((1.f - ax) * d10 + ax * d11);
                const F3 Xs = unproject(cs, u, v, ds);
                float ur, vr;
                project(cam_s, Xs, ur, vr);
                const float dr = depth_in(cam_s, Xs);
                const float ex = ur - fx, ey = vr - fy;
                if (ex * ex + ey * ey < reproj_px * reproj_px && fabsf(dr - d) < rel_depth * d) {
                    ++cnt;
                    sum += dr;
                    if constexpr (VIS) {
                        // floor(u + 1/2) = x0 + (u - x0 >= 1/2), and u - x0 is exact in fp32 (Sterbenz): this rounds the test's own
                        // u with no further rounding.  x0 = w - 1 implies u = w - 1, so the index stays inside the map
                        consistent |= 1u << s;
                        mark_s[s * kBlk + threadIdx.x] = (y0 + (ay >= 0.5f)) * w + x0 + (ax >= 0.5f);
                    }
                }
            }
        }
        keep = valid && cnt >= min_views;
        mask[at] = keep;
        count[at] = cnt;
        fused[at] = sum / (float)(1 + cnt);
        if constexpr (VIS) {
            // several threads may store the same 1 to one byte; no launch writes the used[] slice it reads (the host refuses a
            // view among its own sources), and launches of successive views are ordered on the stream
            if (keep)
                for (unsigned b = consistent; b; b &= b - 1) {
                    const int s = __ffs(b) - 1;
                    used[(size_t)src_s[s] * hw + mark_s[s * kBlk + threadIdx.x]] = 1;
                }
        }
    }
    const int kept = __syncthreads_count(keep);
    if (threadIdx.x == 0) block_counts[(size_t)ref * gridDim.x + blockIdx.x] = kept;
}

__global__ void __launch_bounds__(kBlk) fusion_emit_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ fused,
                                                          const float* __restrict__ colours, const float* __restrict__ cams,
                                                          const int64_t* __restrict__ offsets, int h, int w,
                                                          float* __restrict__ xyz, float* __restrict__ rgb) {
    __shared__ int warp_kept[kBlk / 32];
    const int ref = blockIdx.y, hw = h * w, pix = blockIdx.x * kBlk + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t at = (size_t)ref * hw + pix;
    const bool keep = pix < hw && mask[at];
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_kept[warp] = __popc(bal);
    __syncthreads();
    if (!keep) return;
    int64_t pos = offsets[(size_t)ref * gridDim.x + blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
    for (int i = 0; i < warp; ++i) pos += warp_kept[i];
    const F3 X = unproject(cams + (size_t)ref * kCam, (float)(pix % w), (float)(pix / w), fused[at]);
    xyz[pos * 3 + 0] = X.x;
    xyz[pos * 3 + 1] = X.y;
    xyz[pos * 3 + 2] = X.z;
#pragma unroll
    for (int c = 0; c < 3; ++c) rgb[pos * 3 + c] = colours[((size_t)ref * 3 + c) * hw + pix];
}

__global__ void resize_rgb_kernel(const float* __restrict__ images, int H, int W, int h, int w, float* __restrict__ out) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x, n = blockIdx.y;
    if (pix >= h * w) return;
    const int x = pix % w, y = pix / w;
    const Tap ty = tap_of(y, (float)H / (float)h, H), tx = tap_of(x, (float)W / (float)w, W);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float* p = images + ((size_t)n * 3 + c) * H * W + (size_t)ty.i0 * W + tx.i0;
        const float a = p[0], bq = p[tx.step], cq = p[ty.step * W], d = p[ty.step * W + tx.step];
        out[((size_t)n * 3 + c) * h * w + pix] = ty.l0 * (tx.l0 * a + tx.l1 * bq) + ty.l1 * (tx.l0 * cq + tx.l1 * d);
    }
}

}  // namespace

extern "C" int mvsb200_fusion_check(const float* depth, const float* conf, const float* cams, const int32_t* sources, int N, int S,
                                    int h, int w, float conf_min, float reproj_px, float rel_depth, int min_views,
                                    uint8_t* mask, int32_t* count, float* fused, int32_t* block_counts, void* stream) {
    MVS_REQUIRE(depth && conf && cams && mask && count && fused && block_counts, "fusion_check: null pointer");
    MVS_REQUIRE(S == 0 || sources, "fusion_check: null source table");
    MVS_REQUIRE(N >= 1 && N <= 65535 && h >= 1 && w >= 1 && (long long)h * w < (1LL << 30), "fusion_check: bad shape");
    MVS_REQUIRE(S >= 0 && S <= kMaxSrc, "fusion_check: 0 <= S <= %d sources per view", kMaxSrc);
    dim3 grid((h * w + kBlk - 1) / kBlk, N);
    fusion_check_kernel<false><<<grid, kBlk, 0, (cudaStream_t)stream>>>(depth, conf, cams, sources, S, h, w, conf_min, reproj_px,
                                                                        rel_depth, min_views, mask, count, fused, block_counts, 0,
                                                                        nullptr);
    MVS_CHECK_LAUNCH("fusion_check");
    return MVSB200_OK;
}

extern "C" int mvsb200_fusion_visibility(const float* depth, const float* conf, const float* cams, const int32_t* sources, int N,
                                         int S, int h, int w, float conf_min, float reproj_px, float rel_depth, int min_views, int ref,
                                         uint8_t* used, uint8_t* mask, int32_t* count, float* fused, int32_t* block_counts,
                                         void* stream) {
    MVS_REQUIRE(depth && conf && cams && used && mask && count && fused && block_counts, "fusion_visibility: null pointer");
    MVS_REQUIRE(S == 0 || sources, "fusion_visibility: null source table");
    MVS_REQUIRE(N >= 1 && N <= 65535 && h >= 1 && w >= 1 && (long long)h * w < (1LL << 30), "fusion_visibility: bad shape");
    MVS_REQUIRE(S >= 0 && S <= kMaxSrc, "fusion_visibility: 0 <= S <= %d sources per view", kMaxSrc);
    MVS_REQUIRE(ref >= 0 && ref < N, "fusion_visibility: reference view %d outside [0, %d)", ref, N);
    dim3 grid((h * w + kBlk - 1) / kBlk, 1);
    fusion_check_kernel<true><<<grid, kBlk, 0, (cudaStream_t)stream>>>(depth, conf, cams, sources, S, h, w, conf_min, reproj_px,
                                                                       rel_depth, min_views, mask, count, fused, block_counts, ref,
                                                                       used);
    MVS_CHECK_LAUNCH("fusion_visibility");
    return MVSB200_OK;
}

extern "C" int mvsb200_fusion_emit(const uint8_t* mask, const float* fused, const float* colours, const float* cams,
                                   const int64_t* offsets, int N, int h, int w, float* xyz, float* rgb, void* stream) {
    MVS_REQUIRE(mask && fused && colours && cams && offsets && xyz && rgb, "fusion_emit: null pointer");
    MVS_REQUIRE(N >= 1 && N <= 65535 && h >= 1 && w >= 1 && (long long)h * w < (1LL << 30), "fusion_emit: bad shape");
    dim3 grid((h * w + kBlk - 1) / kBlk, N);
    fusion_emit_kernel<<<grid, kBlk, 0, (cudaStream_t)stream>>>(mask, fused, colours, cams, offsets, h, w, xyz, rgb);
    MVS_CHECK_LAUNCH("fusion_emit");
    return MVSB200_OK;
}

extern "C" int mvsb200_resize_rgb(const float* images, int N, int H, int W, int h, int w, float* out, void* stream) {
    MVS_REQUIRE(images && out, "resize_rgb: null pointer");
    MVS_REQUIRE(N >= 1 && N <= 65535 && H >= 1 && W >= 1 && h >= 1 && w >= 1, "resize_rgb: bad shape");
    dim3 grid((h * w + 127) / 128, N);
    resize_rgb_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(images, H, W, h, w, out);
    MVS_CHECK_LAUNCH("resize_rgb");
    return MVSB200_OK;
}
