// K3c: the regulariser's output convolution, 8 -> 1 channels, k = 3, stride 1, padding 1 (sm_100a, SIMT).
//
// Reference: scripts/model.py:91 `self.conv_out = conv_layer(base_filt, 1, ...)`, used at :123 on (y1 + y0) before the
// depth softmax.  With 8 input channels and ONE output channel this is not a tensor-core shape (K = 8 per tap, N = 1);
// it is 216 MACs per voxel over a 16-byte voxel row -- HBM/L1-bound streaming work.  cuDNN spends 7.3 ms on the forward
// and 13.7 ms on the two gradients at B = 4 (profiles/r01 step profile); these three kernels do the same in ~1 ms.
//   fwd    logits[v]   = sum_tap sum_c W[tap][c] * z[v + tap - 1][c]            z: bf16 [B,D,h,w,8]  ->  fp32 [B,D,h,w]
//   dgrad  gz[v][c]    = sum_tap W[tap][c] * glogits[v - tap + 1]               fp32 [B,D,h,w]       ->  bf16 [B,D,h,w,8]
//   wgrad  gW[tap][c]  = sum_v glogits[v] * z[v + tap - 1][c]                   deterministic two-stage reduction
#include "common.cuh"
#include <stdlib.h>

using namespace mvsb200;

namespace {

constexpr int kCi = 8;
constexpr int kTaps = 27;
constexpr int kWn = kTaps * kCi;                 // 216 filter values

__device__ __forceinline__ void bf16x8_to_f32(const uint4& u, float (&v)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

// ---- forward: one thread per voxel, 32 x 8 (x, y) tiles, one plane per blockIdx.z -------------------------------
__global__ void __launch_bounds__(256) conv_out_fwd_kernel(const uint4* __restrict__ z, const float* __restrict__ wt,
                                                           float* __restrict__ out, int D, int h, int w) {
    __shared__ __align__(16) float s_w[kWn];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    if (tid < kWn) s_w[tid] = wt[tid];
    __syncthreads();
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    const int b = blockIdx.z / D, d = blockIdx.z % D;
    if (x >= w || y >= h) return;
    float acc = 0.f;
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
        const int dz = d + kd - 1;
        if ((unsigned)dz >= (unsigned)D) continue;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
            const int yy = y + kh - 1;
            if ((unsigned)yy >= (unsigned)h) continue;
            const uint4* line = z + ((size_t)(b * D + dz) * h + yy) * w;
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int xx = x + kw - 1;
                if ((unsigned)xx >= (unsigned)w) continue;
                float v[8];
                bf16x8_to_f32(__ldg(line + xx), v);
                const float4 w0 = *reinterpret_cast<const float4*>(s_w + ((kd * 3 + kh) * 3 + kw) * kCi);
                const float4 w1 = *reinterpret_cast<const float4*>(s_w + ((kd * 3 + kh) * 3 + kw) * kCi + 4);
                acc = fmaf(v[0], w0.x, acc); acc = fmaf(v[1], w0.y, acc); acc = fmaf(v[2], w0.z, acc); acc = fmaf(v[3], w0.w, acc);
                acc = fmaf(v[4], w1.x, acc); acc = fmaf(v[5], w1.y, acc); acc = fmaf(v[6], w1.z, acc); acc = fmaf(v[7], w1.w, acc);
            }
        }
    }
    out[((size_t)(b * D + d) * h + y) * w + x] = acc;
}

// ---- data gradient: one thread per voxel ----------------------------------------------------------------------------
__global__ void __launch_bounds__(256) conv_out_dgrad_kernel(const float* __restrict__ g, const float* __restrict__ wt,
                                                             uint4* __restrict__ gz, int D, int h, int w) {
    __shared__ __align__(16) float s_w[kWn];
    const int tid = threadIdx.y * 32 + threadIdx.x;
    if (tid < kWn) s_w[tid] = wt[tid];
    __syncthreads();
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    const int b = blockIdx.z / D, d = blockIdx.z % D;
    if (x >= w || y >= h) return;
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
        const int dz = d - kd + 1;                       // output voxel v - tap + 1 used input voxel v with this tap
        if ((unsigned)dz >= (unsigned)D) continue;
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
            const int yy = y - kh + 1;
            if ((unsigned)yy >= (unsigned)h) continue;
            const float* line = g + ((size_t)(b * D + dz) * h + yy) * w;
#pragma unroll
            for (int kw = 0; kw < 3; ++kw) {
                const int xx = x - kw + 1;
                if ((unsigned)xx >= (unsigned)w) continue;
                const float gv = __ldg(line + xx);
                const float4 w0 = *reinterpret_cast<const float4*>(s_w + ((kd * 3 + kh) * 3 + kw) * kCi);
                const float4 w1 = *reinterpret_cast<const float4*>(s_w + ((kd * 3 + kh) * 3 + kw) * kCi + 4);
                acc[0] = fmaf(gv, w0.x, acc[0]); acc[1] = fmaf(gv, w0.y, acc[1]); acc[2] = fmaf(gv, w0.z, acc[2]); acc[3] = fmaf(gv, w0.w, acc[3]);
                acc[4] = fmaf(gv, w1.x, acc[4]); acc[5] = fmaf(gv, w1.y, acc[5]); acc[6] = fmaf(gv, w1.z, acc[6]); acc[7] = fmaf(gv, w1.w, acc[7]);
            }
        }
    }
    gz[((size_t)(b * D + d) * h + y) * w + x] = make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]),
                                                            pack_bf16x2(acc[4], acc[5]), pack_bf16x2(acc[6], acc[7]));
}

// ---- weight gradient -------------------------------------------------------------------------------------------------
// A warp walks one (b, d, y) line.  Lane = (kw, c) for 24 lanes: it owns the 9 (kd, kh) taps of its (kw, c) and reads, per
// voxel, 9 bf16 values (the 24 lanes of a tap read 48 contiguous bytes) and the broadcast upstream gradient.
constexpr int kWgBlocks = 148 * 4;
__global__ void __launch_bounds__(256) conv_out_wgrad_kernel(const __nv_bfloat16* __restrict__ z, const float* __restrict__ g,
                                                             float* __restrict__ partials, int B, int D, int h, int w) {
    __shared__ float s_acc[8][kWn];                 // one slot per warp: fixed summation order (deterministic)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kw = lane >> 3, c = lane & 7;
    const bool owner = lane < 24;
    float acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    const long lines = (long)B * D * h;
    for (long line = (long)blockIdx.x * 8 + warp; line < lines; line += (long)gridDim.x * 8) {
        const int y = (int)(line % h);
        const int d = (int)((line / h) % D);
        const int b = (int)(line / ((long)h * D));
        const float* gl = g + line * w;
        const __nv_bfloat16* rows[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const int dz = d + t / 3 - 1, yy = y + t % 3 - 1;
            rows[t] = ((unsigned)dz < (unsigned)D && (unsigned)yy < (unsigned)h)
                          ? z + (((size_t)(b * D + dz) * h + yy) * w) * kCi + c : nullptr;
        }
        for (int x = 0; x < w; ++x) {
            const float gv = __ldg(gl + x);
            const int xx = x + kw - 1;
            const bool ok = owner && (unsigned)xx < (unsigned)w;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                if (ok && rows[t] != nullptr) {
                    const float zv = __bfloat162float(rows[t][(size_t)xx * kCi]);
                    acc[t] = fmaf(gv, zv, acc[t]);
                }
            }
        }
    }
    if (owner) {
#pragma unroll
        for (int t = 0; t < 9; ++t) s_acc[warp][(t * 3 + kw) * kCi + c] = acc[t];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kWn; i += 256) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += s_acc[k][i];
        partials[(size_t)blockIdx.x * kWn + i] = s;
    }
}

__global__ void conv_out_wgrad_finalize_kernel(const float* __restrict__ partials, int nblocks, float* __restrict__ gw) {
    const int i = threadIdx.x;
    if (i >= kWn) return;
    double s = 0.0;
    for (int k = 0; k < nblocks; ++k) s += (double)partials[(size_t)k * kWn + i];
    gw[i] = (float)s;
}

// =====================================================================================================================
// Depth-marching forms (the shipped ones).  The one-thread-per-voxel kernels above fetch 27 taps per voxel through L1 and
// read the filter from shared memory (54 LDS.128 per voxel); here a thread owns an (x, y) column and walks a run of planes:
// per INPUT plane it loads the 9 in-plane taps once, forms the three depth-tap partial sums with the filter as
// constant-bank FFMA operands (no load instruction for the weights) and keeps two running sums in registers -- the
// register-level twin of the kdn tensor-core kernel.  The filter lives in one of 8 __constant__ slots, one per launching
// stream (copied device to device on that stream before the kernel: stage_filter).
constexpr int kSlotsW = 8;
__constant__ float c_w[kSlotsW][kWn];
constexpr int kDch = 24;                         // planes per run: (kDch + 2) input planes are visited per kDch outputs

__global__ void __launch_bounds__(256) conv_out_fwd_march_kernel(const uint4* __restrict__ z, float* __restrict__ out, int D, int h,
                                                                 int w, int nch, int slot) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    const int b = blockIdx.z / nch, d0 = (blockIdx.z % nch) * kDch, d1 = min(D, d0 + kDch);
    if (x >= w || y >= h) return;
    const float* cw = c_w[slot];
    bool okx[3], oky[3];
    int offs[9];
#pragma unroll
    for (int k = 0; k < 3; ++k) { okx[k] = (unsigned)(x + k - 1) < (unsigned)w; oky[k] = (unsigned)(y + k - 1) < (unsigned)h; }
#pragma unroll
    for (int t = 0; t < 9; ++t) offs[t] = (min(max(y + t / 3 - 1, 0), h - 1)) * w + min(max(x + t % 3 - 1, 0), w - 1);
    const size_t plane = (size_t)h * w;
    float R1 = 0.f, R2 = 0.f;
    for (int s = d0 - 1; s <= d1; ++s) {
        float p0 = 0.f, p1 = 0.f, p2 = 0.f;
        if ((unsigned)s < (unsigned)D) {
            const uint4* zp = z + (size_t)(b * D + s) * plane;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const bool ok = okx[t % 3] && oky[t / 3];
                uint4 u = __ldg(zp + offs[t]);
                if (!ok) u = make_uint4(0u, 0u, 0u, 0u);
                float v[8];
                bf16x8_to_f32(u, v);
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    p0 = fmaf(v[c], cw[(0 * 9 + t) * kCi + c], p0);
                    p1 = fmaf(v[c], cw[(1 * 9 + t) * kCi + c], p1);
                    p2 = fmaf(v[c], cw[(2 * 9 + t) * kCi + c], p2);
                }
            }
        }
        const float o = R2 + p2;                         // output plane s - 1: taps kd = 0, 1, 2 from input planes s-2, s-1, s
        R2 = R1 + p1;
        R1 = p0;
        if (s - 1 >= d0) out[(size_t)(b * D + s - 1) * plane + (size_t)y * w + x] = o;
    }
}

__global__ void __launch_bounds__(256) conv_out_dgrad_march_kernel(const float* __restrict__ g, uint4* __restrict__ gz, int D, int h,
                                                                   int w, int nch, int slot) {
    const int x = blockIdx.x * 32 + threadIdx.x, y = blockIdx.y * 8 + threadIdx.y;
    const int b = blockIdx.z / nch, d0 = (blockIdx.z % nch) * kDch, d1 = min(D, d0 + kDch);
    if (x >= w || y >= h) return;
    const float* cw = c_w[slot];
    bool okx[3], oky[3];
    int offs[9];
#pragma unroll
    for (int k = 0; k < 3; ++k) { okx[k] = (unsigned)(x - k + 1) < (unsigned)w; oky[k] = (unsigned)(y - k + 1) < (unsigned)h; }
#pragma unroll
    for (int t = 0; t < 9; ++t) offs[t] = (min(max(y - t / 3 + 1, 0), h - 1)) * w + min(max(x - t % 3 + 1, 0), w - 1);
    const size_t plane = (size_t)h * w;
    float R1[8], R2[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { R1[c] = 0.f; R2[c] = 0.f; }
    for (int s = d0 - 1; s <= d1; ++s) {                 // planes of the upstream gradient
        float q0[8], q1[8], q2[8];                       // its contribution to output planes s-1 (kd=0), s (kd=1), s+1 (kd=2)
#pragma unroll
        for (int c = 0; c < 8; ++c) { q0[c] = 0.f; q1[c] = 0.f; q2[c] = 0.f; }
        if ((unsigned)s < (unsigned)D) {
            const float* gp = g + (size_t)(b * D + s) * plane;
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const bool ok = okx[t % 3] && oky[t / 3];
                float gv = __ldg(gp + offs[t]);
                if (!ok) gv = 0.f;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    q0[c] = fmaf(gv, cw[(0 * 9 + t) * kCi + c], q0[c]);
                    q1[c] = fmaf(gv, cw[(1 * 9 + t) * kCi + c], q1[c]);
                    q2[c] = fmaf(gv, cw[(2 * 9 + t) * kCi + c], q2[c]);
                }
            }
        }
        float o[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) { o[c] = R2[c] + q0[c]; R2[c] = R1[c] + q1[c]; R1[c] = q2[c]; }
        if (s - 1 >= d0)
            gz[(size_t)(b * D + s - 1) * plane + (size_t)y * w + x] =
                make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
    }
}

// Weight gradient, depth-marching form.  gW[tap][c] = sum_v g[v] * z[v + tap - 1][c]  ==  every z voxel u adds
// z[u][c] * g[u - (tap - 1)] to the 27 taps.  A thread owns an (x, y) column and TWO channels (4 threads per voxel, a warp = 8
// pixels of a line) and walks a run of planes: per plane it loads its 4 bytes of the voxel row once and multiplies them into 27
// accumulator pairs with the 3x3x3 neighbourhood of g -- three planes of 9 values held in registers (rotated by unrolling the
// plane loop three times), the entering plane read through L1 (the 4 threads of a pixel and the 8 pixels of a warp share the
// lines).  54 FMAs per 4 bytes of z instead of 8 per 16 bytes and tap (the previous form: a warp per line, lane = tap, 22
// instructions per 216 MACs); no shared memory, no barrier in the loop (a first version staged g through a shared tile with
// two CTA barriers per plane: 1.0 ms instead of 0.7 -- barrier bound).  CTAs are persistent (one wave): accumulators run on
// across work items and are reduced once (shuffles in a fixed order, then the deterministic finalize).
constexpr int kWTX = 16, kWTY = 4, kWDchunk = 48;    // pixel tile, planes per work item (a multiple of 3)
constexpr int kWgMarchCtasPerSm = 2;                // persistent grid: CTAs per SM, the residency of __launch_bounds__(256, 2)
__device__ float c_zero_row[4];                      // where the row pointer of a line outside the image points

__global__ void __launch_bounds__(256, 2) conv_out_wgrad_march_kernel(const uint32_t* __restrict__ z, const float* __restrict__ g,
                                                                      float* __restrict__ partials, int B, int D, int h, int w,
                                                                      int tiles_x, int tiles_y, int nchunks, int n_items) {
    __shared__ float s_red[8][4][54];                // per warp, per channel pair
    const int tid = threadIdx.x, cp = tid & 3, pix = tid >> 2;
    const int lx = pix & (kWTX - 1), ly = pix / kWTX;
    float2 acc[27];
#pragma unroll
    for (int t = 0; t < 27; ++t) acc[t] = make_float2(0.f, 0.f);
    const size_t plane = (size_t)h * w;

    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int t = item % (tiles_x * tiles_y), r = item / (tiles_x * tiles_y);
        const int c = r % nchunks, b = r / nchunks;
        const int d0 = c * kWDchunk, nd = min(kWDchunk, D - d0);
        const int x = (t % tiles_x) * kWTX + lx, y = (t / tiles_x) * kWTY + ly;
        const bool inside = x < w && y < h;
        const float* gb = g + (size_t)b * D * plane;
        // in-plane neighbours g[.][y - kh + 1][x - kw + 1].  Address arithmetic is what this loop must not do (a first
        // barrier-free version spent ~250 of its 280 instructions per plane on 64-bit address generation and predicates for
        // nine guarded loads): per item one row pointer per kh (a row outside the image points at a zero word and never
        // advances), per plane one multiply-add per row, the three kw taps at fixed element offsets (0 where the column is
        // outside the image, the loaded value then replaced by 0)
        const float* rowp[3];
        long long rstep[3];
        int offx[3];
        bool colok[3];
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
            const int xx = x - kw + 1;
            colok[kw] = inside && (unsigned)xx < (unsigned)w;
            offx[kw] = colok[kw] ? 1 - kw : 0;
        }
#pragma unroll
        for (int kh = 0; kh < 3; ++kh) {
            const int yy = y - kh + 1;
            const bool rok = inside && (unsigned)yy < (unsigned)h;
            rowp[kh] = rok ? gb + (size_t)yy * w + x : c_zero_row;
            rstep[kh] = rok ? (long long)plane : 0;
        }
        auto read_plane = [&](int p, float (&dst)[9]) {          // plane p of g, zero outside the volume
            const int pc = min(max(p, 0), D - 1);
#pragma unroll
            for (int kh = 0; kh < 3; ++kh) {
                const float* rp = rowp[kh] + rstep[kh] * pc;
#pragma unroll
                for (int kw = 0; kw < 3; ++kw) {
                    const float v = __ldg(rp + offx[kw]);
                    dst[kh * 3 + kw] = colok[kw] ? v : 0.f;
                }
            }
            if (p != pc) {                            // uniform over the CTA: the plane below / above the volume
#pragma unroll
                for (int k9 = 0; k9 < 9; ++k9) dst[k9] = 0.f;
            }
        };
        float g0[9], g1[9], g2[9];                    // planes d-1, d, d+1 of the current step (roles rotate)
        read_plane(d0 - 1, g0);
        read_plane(d0, g1);
        const uint32_t* zc = z + (((size_t)b * D + d0) * plane + (size_t)y * w + x) * 4 + cp;     // 4 channel pairs per voxel row
        const size_t zstep = plane * 4;
        auto step = [&](int dd, const float (&lo)[9], const float (&mid)[9], float (&hi)[9]) {
            read_plane(d0 + dd + 1, hi);
            float2 zv = make_float2(0.f, 0.f);
            if (inside && dd < nd) {
                const uint32_t u = __ldg(zc);
                zv = make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
            }
            zc += zstep;
            // tap (kd, kh, kw) pairs z[d] with g at plane d - kd + 1: kd = 0 -> hi, 1 -> mid, 2 -> lo
#pragma unroll
            for (int k9 = 0; k9 < 9; ++k9) {
                acc[k9] = __ffma2_rn(make_float2(hi[k9], hi[k9]), zv, acc[k9]);
                acc[9 + k9] = __ffma2_rn(make_float2(mid[k9], mid[k9]), zv, acc[9 + k9]);
                acc[18 + k9] = __ffma2_rn(make_float2(lo[k9], lo[k9]), zv, acc[18 + k9]);
            }
        };
        for (int dd = 0; dd < nd; dd += 3) {          // planes beyond nd contribute zero (zv = 0)
            step(dd, g0, g1, g2);
            step(dd + 1, g1, g2, g0);
            step(dd + 2, g2, g0, g1);
        }
    }
    // reduce over the pixels of the CTA, fixed order: lanes of a warp with the same channel pair (xor 4, 8, 16), then warps
#pragma unroll
    for (int t = 0; t < 27; ++t) {
#pragma unroll
        for (int m = 4; m < 32; m <<= 1) {
            acc[t].x += __shfl_xor_sync(0xffffffffu, acc[t].x, m);
            acc[t].y += __shfl_xor_sync(0xffffffffu, acc[t].y, m);
        }
    }
    const int lane = tid & 31, warp = tid >> 5;
    if (lane < 4) {
#pragma unroll
        for (int t = 0; t < 27; ++t) { s_red[warp][lane][2 * t] = acc[t].x; s_red[warp][lane][2 * t + 1] = acc[t].y; }
    }
    __syncthreads();
    for (int i = tid; i < kWn; i += 256) {           // i = tap * 8 + channel
        const int tap = i >> 3, ch = i & 7;
        float sum = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) sum += s_red[k][ch >> 1][2 * tap + (ch & 1)];
        partials[(size_t)blockIdx.x * kWn + i] = sum;
    }
}

// One filter slot per launching stream (first come, first served): a stream's staging copy and its kernels are ordered, and
// two streams -- or a replaying graph captured on its own stream beside eager launches -- never overwrite a slot under each
// other's live kernel.  More than kSlotsW distinct streams share the last slot (single-stream ordering still holds there).
int stage_filter(const float* w27x8, cudaStream_t st, int* slot_out) {
    static std::atomic<uintptr_t> owner[kSlotsW];
    const uintptr_t id = reinterpret_cast<uintptr_t>(st) + 1;          // +1: the default stream (0) is an owner too
    int slot = kSlotsW - 1;
    for (int i = 0; i < kSlotsW; ++i) {
        uintptr_t cur = owner[i].load(std::memory_order_acquire);
        if (cur == 0 && owner[i].compare_exchange_strong(cur, id)) cur = id;
        if (cur == id) { slot = i; break; }
    }
    MVS_CUDA(cudaMemcpyToSymbolAsync(c_w, w27x8, sizeof(float) * kWn, sizeof(float) * kWn * slot, cudaMemcpyDeviceToDevice, st));
    *slot_out = slot;
    return MVSB200_OK;
}

bool use_march() {
    const char* e = getenv("MVSB200_CONV_OUT");
    return !(e && e[0] == 'v');                          // MVSB200_CONV_OUT=voxel selects the one-thread-per-voxel kernels
}

int check_shape(int B, int D, int h, int w, const char* name) {
    MVS_REQUIRE(B >= 1 && D >= 1 && h >= 1 && w >= 1 && (long)B * D <= 65535 && (h + 7) / 8 <= 65535 && (long)h * w < (1L << 30),
                "%s: bad shape", name);
    return MVSB200_OK;
}

}  // namespace

extern "C" int64_t mvsb200_conv_out_workspace_floats(void) { return (int64_t)kWgBlocks * kWn; }

extern "C" int mvsb200_conv_out_fwd(const void* z, const float* w27x8, float* logits, int B, int D, int h, int w, void* stream) {
    MVS_REQUIRE(z && w27x8 && logits && aligned16(z), "conv_out_fwd: null or misaligned pointer");
    if (int rc = check_shape(B, D, h, w, "conv_out_fwd")) return rc;
    if (use_march()) {
        int slot = 0;
        if (int rc = stage_filter(w27x8, (cudaStream_t)stream, &slot)) return rc;
        const int nch = (D + kDch - 1) / kDch;
        const dim3 grid((w + 31) / 32, (h + 7) / 8, B * nch);
        conv_out_fwd_march_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>((const uint4*)z, logits, D, h, w, nch, slot);
        MVS_CHECK_LAUNCH("conv_out_fwd_march");
        return MVSB200_OK;
    }
    const dim3 grid((w + 31) / 32, (h + 7) / 8, B * D);
    conv_out_fwd_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>((const uint4*)z, w27x8, logits, D, h, w);
    MVS_CHECK_LAUNCH("conv_out_fwd");
    return MVSB200_OK;
}

extern "C" int mvsb200_conv_out_dgrad(const float* glogits, const float* w27x8, void* gz, int B, int D, int h, int w, void* stream) {
    MVS_REQUIRE(glogits && w27x8 && gz && aligned16(gz), "conv_out_dgrad: null or misaligned pointer");
    if (int rc = check_shape(B, D, h, w, "conv_out_dgrad")) return rc;
    if (use_march()) {
        int slot = 0;
        if (int rc = stage_filter(w27x8, (cudaStream_t)stream, &slot)) return rc;
        const int nch = (D + kDch - 1) / kDch;
        const dim3 grid((w + 31) / 32, (h + 7) / 8, B * nch);
        conv_out_dgrad_march_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(glogits, (uint4*)gz, D, h, w, nch, slot);
        MVS_CHECK_LAUNCH("conv_out_dgrad_march");
        return MVSB200_OK;
    }
    const dim3 grid((w + 31) / 32, (h + 7) / 8, B * D);
    conv_out_dgrad_kernel<<<grid, dim3(32, 8), 0, (cudaStream_t)stream>>>(glogits, w27x8, (uint4*)gz, D, h, w);
    MVS_CHECK_LAUNCH("conv_out_dgrad");
    return MVSB200_OK;
}

extern "C" int mvsb200_conv_out_wgrad(const void* z, const float* glogits, float* workspace, float* gw27x8, int B, int D, int h,
                                      int w, void* stream) {
    MVS_REQUIRE(z && glogits && workspace && gw27x8, "conv_out_wgrad: null pointer");
    if (int rc = check_shape(B, D, h, w, "conv_out_wgrad")) return rc;
    const long lines = (long)B * D * h;
    const int blocks = (int)((lines + 7) / 8 < kWgBlocks ? (lines + 7) / 8 : kWgBlocks);
    if (use_march()) {
        MVS_REQUIRE(aligned16(z), "conv_out_wgrad: misaligned volume");
        const int tiles_x = (w + kWTX - 1) / kWTX, tiles_y = (h + kWTY - 1) / kWTY, nchunks = (D + kWDchunk - 1) / kWDchunk;
        const long items = (long)tiles_x * tiles_y * nchunks * B;
        MVS_REQUIRE(items < (1L << 31), "conv_out_wgrad: volume too large");
        // the persistent grid is one wave: as many CTAs as the device holds at once (2 per SM at 128 registers x 256 threads),
        // taken from the device's SM count.  One CTA per SM would leave half of every SM to the streaming kernels the side
        // stream's weight gradient runs beside (mvs_b200/ops.py, wgrad_fork), but measured slower in the cfg2 step: 15.97
        // against 15.57 ms (profiles/r07_wgrad_overlap.md)
        const int sms = sm_count();
        const long cap = (long)kWgMarchCtasPerSm * sms < kWgBlocks ? (long)kWgMarchCtasPerSm * sms : kWgBlocks;
        const int grid = (int)(items < cap ? items : cap);
        conv_out_wgrad_march_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint32_t*)z, glogits, workspace, B, D, h, w, tiles_x,
                                                                            tiles_y, nchunks, (int)items);
        MVS_CHECK_LAUNCH("conv_out_wgrad_march");
        conv_out_wgrad_finalize_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(workspace, grid, gw27x8);
        MVS_CHECK_LAUNCH("conv_out_wgrad_finalize");
        return MVSB200_OK;
    } else {
        conv_out_wgrad_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)z, glogits, workspace, B, D, h, w);
        MVS_CHECK_LAUNCH("conv_out_wgrad");
    }
    conv_out_wgrad_finalize_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(workspace, blocks, gw27x8);
    MVS_CHECK_LAUNCH("conv_out_wgrad_finalize");
    return MVSB200_OK;
}
