// K3 (backward of the stride-2 layers): weight gradient of the stride-2 convolutions and of the stride-2 transposed
// convolutions of the regulariser on tcgen05 tensor cores, ONE launch per layer (sm_100a).
//
// Reference semantics (citations into /root/reference/scripts):
//   model.py:104-110   conv_{1,2,3}_0 = Conv3d(k=3, stride=2, padding=dim/2+1)          big = layer input, small = output gradient
//   model.py:115-121   deconv_{3,2,1}_0 = ConvTranspose3d(k=3, stride=2, ...)           big = output gradient, small = layer input
//   model.py:223-234   the factories; autograd's weight gradient of both is
//       gw[k][cb][cs] = sum_{b,o} big(2o - pad + k)[cb] * small(o)[cs]     k = (kd,kh,kw), big zero outside its volume.
//
// GEMM view: the reduction runs over voxels, so both operands are MN-major (voxel = K row, channels contiguous).  The
// stride-2 read of `big` along w is removed WITHOUT de-interleaving copies: a TMA tensor map presents each line of `big` as
// rows of voxel PAIRS (2*Cb channels per row = one swizzle atom); output voxel ox needs the pairs ox-1 and ox, and an
// MN-major operand may be assembled from swizzle atoms that start at ANY row, so
//     A[K = ox, M = (pair a in {ox-1, ox}, w parity, cb)]   = the pair-row line read from row ox, atoms one row apart
//     B[K = ox, N = cs]                                     = the matching line of `small`
// and one tcgen05.mma chain over a line accumulates all three kw taps of one (kd, kh):  three of the four (a, parity)
// row groups of D are the taps kw = 2(a-1) + parity + pad, the fourth is dropped.  Lines of `big` are addressed directly
// (y = 2 oy - pad + kh, d = 2 od - pad + kd): no de-interleaving along h or depth is needed because a line is the unit.
// A CTA owns ONE depth tap kd (blockIdx % 3) and keeps its three kh accumulator blocks (3 x Cs fp32 columns) in TMEM over
// its whole life.  The TMA producer and the MMA issuer are single-warp serial code, so the pipeline is organised to cost ONE
// barrier wait, ONE expect_tx and ONE commit per line of small (measured: with a barrier per loaded line and run-time
// modulo ring indices the kernel took 0.9 ms whatever the channel counts, MMAs and loads switched off -- the skeleton was
// the bound): a ring STAGE holds a line of small and the two new lines of big it needs (kh = 1, 2; kh = 0 is the previous
// stage's kh = 2 line, or a third line loaded with the first stage of an item).  The three kd CTAs of the same rank walk the
// same lines of `small` at the same time (L2 hits).  Epilogue: fp32 vector reductions into gw.
#include "tc_common.cuh"
#include <stdlib.h>

using namespace mvsb200;

namespace {

constexpr int kWgThreads = 192;
constexpr int kMaxRing = 8;
constexpr int kZeroA = 4096;        // zero operand for the accumulator-initialising MMA: 16 + 8 rows of <= 128 bytes ...
constexpr int kZeroB = 4096;        // ... and two N atoms of 16 rows x 128 bytes, 2048 bytes apart

struct S2WgLineParams {
    int B, Ds, Hs, Ws;              // small volume
    int Db, Hb;                     // planes / lines of big
    int pad_d, pad_h, pad_w;
    int Cs;                         // channels of small = MMA N
    int n_chunks, chunk_ch;         // small is loaded as n_chunks boxes of chunk_ch channels (one swizzle atom each)
    int ksteps;                     // ceil(Ws / 16)
    int line_a_bytes, line_b_bytes; // ring slot of a big line; one chunk of a small line (= stride between its N atoms)
    int stage_bytes, n_stages;      // stage = [small: n_chunks x line_b_bytes] then per depth tap of the CTA [big kh=0][kh=1][kh=2]
    int nkd;                        // depth taps per CTA: 1 (blockIdx % 3 picks it) or 3 (narrow layers: 9 x Cs columns fit TMEM,
                                    // a third of the barrier round trips per MMA)
    int ychunk, nychunks;           // lines of small per item
    float* gw;                      // [27][CB][Cs] fp32, accumulated into
    int dbg;                        // diagnostics (MVSB200_S2WG_DBG): 1 = no MMAs issued, 2 = no TMA loads issued
};

// MN-major operand descriptor with the row pitch (= swizzle span) given at run time
__device__ __forceinline__ uint64_t umma_desc_mn_rt(uint32_t saddr, uint32_t rowb, uint32_t atom_stride) {
    const uint64_t layout = rowb == 128 ? 2 : (rowb == 64 ? 4 : 6);
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)((atom_stride >> 4) & 0x3fff) << 16;   // LBO = stride between MN atoms
    d |= (uint64_t)((8 * rowb) >> 4) << 32;               // SBO = stride between 8-row K groups
    d |= (uint64_t)1 << 46;
    d |= layout << 61;
    return d;
}

__device__ __forceinline__ void red_add_v4(float* p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int CB>
__global__ void __launch_bounds__(kWgThreads, 1)
conv3d_s2_wgrad_lines_kernel(const __grid_constant__ CUtensorMap tm_big, const __grid_constant__ CUtensorMap tm_small,
                             const __grid_constant__ S2WgLineParams p) {
    constexpr int ROWA = 4 * CB;                        // bytes of a voxel-pair row == swizzle span of A
    constexpr int ATOM_ROWS = 2 * CB;                   // D rows per atom: (w parity, cb)
    const int ROWG = 2 * p.chunk_ch;                    // bytes of a row of a small chunk == swizzle span of B
    // D fp32, A/B bf16, A and B MN-major, N = Cs, M = 128
    const uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(p.Cs >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* zero_a = smem;
    unsigned char* zero_b = smem + kZeroA;
    unsigned char* stages = zero_b + kZeroB;
    const int slot_b_bytes = p.n_chunks * p.line_b_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(stages + (size_t)p.n_stages * p.stage_bytes);
    uint64_t* full = bars;                      // [kMaxRing]  stage landed
    uint64_t* empty = bars + kMaxRing;          // [kMaxRing]  stage no longer read by any MMA
    uint64_t* done = bars + 2 * kMaxRing;       // [1]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkd = p.nkd;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 3 * nkd * p.Cs) tmem_cols <<= 1;

    // zero everything the MMAs may read and TMA never writes: the zero operands, the row tails of every ring slot
    {
        uint4* z = reinterpret_cast<uint4*>(smem);
        const int n = (int)((reinterpret_cast<unsigned char*>(bars) - smem) / 16);
        for (int i = threadIdx.x; i < n; i += kWgThreads) z[i] = make_uint4(0, 0, 0, 0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_big) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_small) : "memory");
        for (int i = 0; i < kMaxRing; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        mbar_init(done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // this CTA's depth tap(s) and its share of the (batch, plane of small, line chunk) items
    const int kd0 = nkd == 1 ? (int)blockIdx.x % 3 : 0;
    const int rank = nkd == 1 ? (int)blockIdx.x / 3 : (int)blockIdx.x;
    const int nrank = nkd == 1 ? ((int)gridDim.x - kd0 + 2) / 3 : (int)gridDim.x;
    const int od_lo = nkd == 1 ? max(0, (p.pad_d - kd0 + 1) >> 1) : 0;
    const int od_hi = nkd == 1 ? min(p.Ds - 1, (p.Db - 1 + p.pad_d - kd0) >> 1) : p.Ds - 1;
    const int nod = max(0, od_hi - od_lo + 1);
    const int n_items = p.B * nod * p.nychunks;

    // item -> (b, od, d of the CTA's first depth tap, [oy0, oy1)); depth tap kd0 + i reads plane d + i
    auto decode = [&](int item, int& b, int& od, int& d, int& oy0, int& oy1) {
        const int yc = item % p.nychunks, r = item / p.nychunks;
        od = od_lo + r % nod;
        b = r / nod;
        d = 2 * od - p.pad_d + kd0;
        oy0 = yc * p.ychunk;
        oy1 = min(p.Hs, oy0 + p.ychunk);
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        const uint32_t bytes_a = (uint32_t)ROWA * (p.Ws + 1);
        const uint32_t bytes_b = (uint32_t)ROWG * p.Ws * p.n_chunks;
        int slot = 0, round = 0;                         // ring position of the next stage, times the ring has wrapped
        for (int item = rank; item < n_items; item += nrank) {
            int b, od, d, oy0, oy1;
            decode(item, b, od, d, oy0, oy1);
            for (int oy = oy0; oy < oy1; ++oy) {
                if (round > 0) mbar_wait(empty + slot, (round - 1) & 1);
                if (elect_one()) {
                    unsigned char* st = stages + (size_t)slot * p.stage_bytes;
                    const int y0 = 2 * oy - p.pad_h;
                    const int kh_first = oy == oy0 ? 0 : 1;          // kh = 0 of later lines is the previous stage's kh = 2 line
                    uint32_t bytes = bytes_b;
                    for (int i = 0; i < nkd; ++i)
                        if (d + i >= 0 && d + i < p.Db)
                            for (int kh = kh_first; kh < 3; ++kh) bytes += (y0 + kh >= 0 && y0 + kh < p.Hb) ? bytes_a : 0u;
                    if (p.dbg & 2) { mbar_arrive(full + slot); }
                    else {
                        mbar_expect_tx(full + slot, bytes);
                        for (int c = 0; c < p.n_chunks; ++c)
                            tma_load_5d(st + (size_t)c * p.line_b_bytes, &tm_small, full + slot, c * p.chunk_ch, 0, oy, od, b);
                        // pairs -1 .. Ws-1 of a line of big: smem row r holds pair r - 1 (pair -1 and pairs beyond the line: zeros)
                        for (int i = 0; i < nkd; ++i)
                            if (d + i >= 0 && d + i < p.Db)
                                for (int kh = kh_first; kh < 3; ++kh)
                                    if (y0 + kh >= 0 && y0 + kh < p.Hb)
                                        tma_load_5d(st + slot_b_bytes + (size_t)(i * 3 + kh) * p.line_a_bytes, &tm_big, full + slot, 0, -1,
                                                    y0 + kh, d + i, b);
                    }
                }
                __syncwarp();
                if (++slot == p.n_stages) { slot = 0; ++round; }
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        const uint64_t da0 = umma_desc_mn<ROWA>(0, ROWA);                                   // A atoms: one pair row apart
        const uint64_t db0 = umma_desc_mn_rt(0, (uint32_t)ROWG, (uint32_t)p.line_b_bytes);  // B atoms: one chunk apart
        const uint64_t dz0 = umma_desc_mn_rt(0, (uint32_t)ROWG, 2048u);
        const uint32_t a_hi = (uint32_t)(da0 >> 32), b_hi = (uint32_t)(db0 >> 32), z_hi = (uint32_t)(dz0 >> 32);
        const uint32_t sa_lo = (uint32_t)da0 | (smem_u32(stages) >> 4);
        const uint32_t sb_lo = (uint32_t)db0 | (smem_u32(stages) >> 4);
        const uint32_t st16 = (uint32_t)p.stage_bytes >> 4, la16 = (uint32_t)p.line_a_bytes >> 4, big16 = (uint32_t)slot_b_bytes >> 4;
        // the accumulator blocks (depth tap, kh) start at zero: one MMA each on the all-zero operands
        if (elect_one()) {
            for (int kh = 0; kh < 3 * nkd; ++kh)
                umma_bf16_lohi(tmem_base + (uint32_t)(kh * p.Cs), (uint32_t)da0 | (smem_u32(zero_a) >> 4), a_hi,
                               (uint32_t)dz0 | (smem_u32(zero_b) >> 4), z_hi, IDESC, 0u);
        }
        __syncwarp();
        int slot = 0, round = 0, prev = 0;
        for (int item = rank; item < n_items; item += nrank) {
            int b, od, d, oy0, oy1;
            decode(item, b, od, d, oy0, oy1);
            for (int oy = oy0; oy < oy1; ++oy) {
                mbar_wait(full + slot, round & 1);
                tc_fence_after();
                if (elect_one()) {
                    const int y0 = 2 * oy - p.pad_h;
                    const uint32_t g_lo = sb_lo + (uint32_t)slot * st16;
                    for (int i = 0; i < nkd; ++i) {
                        if (d + i < 0 || d + i >= p.Db) continue;
                        for (int kh = 0; kh < 3; ++kh) {
                            if (y0 + kh < 0 || y0 + kh >= p.Hb) continue;
                            const uint32_t d_tmem = tmem_base + (uint32_t)((i * 3 + kh) * p.Cs);
                            uint32_t a_lo = (kh == 0 && oy != oy0) ? sa_lo + (uint32_t)prev * st16 + big16 + (uint32_t)(i * 3 + 2) * la16
                                                                   : sa_lo + (uint32_t)slot * st16 + big16 + (uint32_t)(i * 3 + kh) * la16;
                            uint32_t b_lo = g_lo;
                            if (p.dbg & 1) continue;
#pragma unroll 2
                            for (int ks = 0; ks < p.ksteps; ++ks) {
                                umma_bf16_lohi(d_tmem, a_lo, a_hi, b_lo, b_hi, IDESC, 1u);
                                a_lo += (uint32_t)(16 * ROWA) >> 4;
                                b_lo += (uint32_t)(16 * ROWG) >> 4;
                            }
                        }
                    }
                    if (oy != oy0) umma_commit(empty + prev);        // its kh = 2 line was this line's kh = 0
                    if (oy == oy1 - 1) umma_commit(empty + slot);
                }
                __syncwarp();
                prev = slot;
                if (++slot == p.n_stages) { slot = 0; ++round; }
            }
        }
        if (elect_one()) umma_commit(done);
        __syncwarp();
    } else {
        // ===================================== epilogue: TMEM -> gw ==============================
        mbar_wait(done, 0);
        tc_fence_after();
        const int q = warp & 3;
        const int m = q * 32 + lane;                     // D row = (pair atom a, w parity, cb)
        const int a = m / ATOM_ROWS, par = (m / CB) & 1, cb = m % CB;
        const int kw = 2 * (a - 1) + par + p.pad_w;      // pair ox + a - 1, voxel 2(ox + a - 1) + par = 2 ox - pad + kw
        const bool real = kw >= 0 && kw <= 2 && n_items > 0;
        for (int blk = 0; blk < 3 * nkd; ++blk) {
            const int kd = kd0 + blk / 3, kh = blk % 3;
            float* dst = p.gw + ((size_t)(((kd * 3 + kh) * 3 + (real ? kw : 0)) * CB + cb)) * p.Cs;
            for (int c0 = 0; c0 < p.Cs; c0 += 16) {
                uint32_t v[16];
                tmem_ld<16>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(blk * p.Cs + c0), v);
                tmem_ld_wait();
                if (real) {
#pragma unroll
                    for (int k = 0; k < 16; k += 4)
                        red_add_v4(dst + c0 + k, __uint_as_float(v[k]), __uint_as_float(v[k + 1]), __uint_as_float(v[k + 2]),
                                   __uint_as_float(v[k + 3]));
                }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

template <int CB>
int launch_s2_wgrad_lines(const void* big, const void* small, float* gw, int B, int Db, int Hb, int Wb, int Ds, int Hs, int Ws,
                          int Cs, int pad_d, int pad_h, int pad_w, const long long* ss, cudaStream_t st) {
    constexpr int ROWA = 4 * CB;
    constexpr int ATOMS = 128 / (2 * CB);
    S2WgLineParams p;
    p.B = B; p.Ds = Ds; p.Hs = Hs; p.Ws = Ws; p.Db = Db; p.Hb = Hb;
    p.pad_d = pad_d; p.pad_h = pad_h; p.pad_w = pad_w;
    p.Cs = Cs;
    p.n_chunks = Cs > 64 ? 2 : 1;
    p.chunk_ch = Cs > 64 ? 64 : Cs;
    const int ROWG = 2 * p.chunk_ch;
    p.ksteps = (Ws + 15) / 16;
    const int rows_a = (Ws + 1 > 16 * p.ksteps + ATOMS ? Ws + 1 : 16 * p.ksteps + ATOMS);
    p.line_a_bytes = (rows_a * ROWA + 1023) / 1024 * 1024;
    p.line_b_bytes = (16 * p.ksteps * ROWG + 1023) / 1024 * 1024;
    const size_t budget = 227 * 1024 - 1024 - kZeroA - kZeroB - 512;
    const size_t slot_b = (size_t)p.n_chunks * p.line_b_bytes;
    // narrow layers: all three depth taps in one CTA when their 9 x Cs accumulator columns fit TMEM and three stages fit shared
    // memory (a third of the barrier round trips per MMA: the small-channel layers are bound by the single-warp roles)
    p.nkd = (9 * Cs <= 512 && 3 * (slot_b + 9 * (size_t)p.line_a_bytes) <= budget) ? 3 : 1;
    if (const char* e = getenv("MVSB200_S2WG_NKD")) { const int v = atoi(e); if (v == 1 || (v == 3 && 9 * Cs <= 512)) p.nkd = v; }
    p.stage_bytes = (int)slot_b + 3 * p.nkd * p.line_a_bytes;
    p.n_stages = (int)(budget / (size_t)p.stage_bytes);
    if (p.n_stages > kMaxRing) p.n_stages = kMaxRing;
    MVS_REQUIRE(p.n_stages >= 2, "conv3d_s2_wgrad_lines: lines of %d voxels do not fit shared memory (Cb=%d, Cs=%d)", Ws, CB, Cs);

    CUtensorMap tm_big, tm_small;
    // big as rows of voxel pairs (Wb is even): 2 * CB channels, Wb / 2 rows per line
    MVS_TRY(encode_volume(&tm_big, big, 2 * CB, 2 * CB, Wb / 2, Hb, Db, B, Ws + 1, 1, "conv3d_s2_wgrad_lines", "big"));
    {
        // voxel-row strides of small in bytes: dense channel-last, or those of the allocation the box lives in (ss: elements)
        const cuuint64_t rowb = (cuuint64_t)2 * Cs;
        const cuuint64_t dims[5] = {(cuuint64_t)Cs, (cuuint64_t)Ws, (cuuint64_t)Hs, (cuuint64_t)Ds, (cuuint64_t)B};
        const cuuint64_t dense[4] = {rowb, rowb * Ws, rowb * Ws * Hs, rowb * Ws * Hs * Ds};
        const cuuint64_t strides[4] = {ss ? (cuuint64_t)ss[3] * 2 : dense[0], ss ? (cuuint64_t)ss[2] * 2 : dense[1],
                                       ss ? (cuuint64_t)ss[1] * 2 : dense[2], ss ? (cuuint64_t)ss[0] * 2 : dense[3]};
        const cuuint32_t box[5] = {(cuuint32_t)p.chunk_ch, (cuuint32_t)Ws, 1, 1, 1};
        MVS_TRY(encode_tiled(&tm_small, small, 5, dims, strides, box, swizzle_for(ROWG), "conv3d_s2_wgrad_lines", "small"));
    }
    int sms = sm_count();
    if (sms < 3) sms = 3;
    // lines of small per item: balance (items per CTA of a depth tap) x (lines + the extra big lines at an item's start)
    const long nrank = p.nkd == 1 ? sms / 3 : sms;
    const Runs runs = choose_runs(Ds, B, Hs, nrank, 2);
    p.nychunks = runs.nchunks;
    p.ychunk = runs.chunk;
    p.gw = gw;
    p.dbg = 0;
    if (const char* e = getenv("MVSB200_S2WG_DBG")) p.dbg = atoi(e);
    if (p.dbg & 4) fprintf(stderr, "s2wg: CB=%d Cs=%d ksteps=%d line_a=%d line_b=%d stage=%d n_stages=%d nyc=%d ychunk=%d\n", CB, Cs, p.ksteps, p.line_a_bytes, p.line_b_bytes, p.stage_bytes, p.n_stages, p.nychunks, p.ychunk);
    const size_t smem = 1024 + kZeroA + kZeroB + (size_t)p.n_stages * p.stage_bytes + 512;
    MVS_CUDA(cudaFuncSetAttribute(conv3d_s2_wgrad_lines_kernel<CB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv3d_s2_wgrad_lines_kernel<CB><<<dim3((unsigned)sms), kWgThreads, smem, st>>>(tm_big, tm_small, p);
    MVS_CHECK_LAUNCH("conv3d_s2_wgrad_lines");
    return MVSB200_OK;
}


// =================================================================================================================
// Data gradient of the stacked stride-2 branches conv_{1,2,3}_0 (scripts/model.py:104-110): with the forward
//   out(o)[co] = sum_k W[k][co][ci] x(2o - pad + k)[ci],   co over the 16 + 32 + 64 = 112 stacked output channels,
// the gradient is the stride-2 TRANSPOSED convolution of the 112-channel box gradient onto the 32-channel canvas
//   gx[2J + par] = sum over the taps k with (par + pad - k) even of W[k]^T . gy[J + (par + pad - k)/2]        (per axis).
// Same skeleton as deconv3d_s2_tc_kernel (conv3d_tc.cu): a CTA marches along depth, the 8 output-parity classes sit side by
// side in TMEM and are written interleaved.  What is new:
//   * K = 112 is not a swizzle span, and a 27-tap filter of 112 x 32 does not fit shared memory next to the slabs.  The
//     contraction runs over K CHUNKS of 16 / 32 / 64 channels -- exactly the three branches -- each its own TMA map, swizzle
//     mode and UMMA descriptor (rows of 32 / 64 / 128 bytes: 224 bytes per voxel, no padding), and the OUTPUT channels are
//     split in halves of NOUT = 16 over NEIGHBOURING CTAs of one launch (blockIdx & 1): the two CTAs walk the same items at
//     the same time, so the slab loads of the second hit L2 and the two 32-byte halves of an output voxel row meet in L2.
//   * ONE MMA PER INPUT SHIFT (DeconvWide, tc_common.cuh): 8 MMAs per K step, classes in Gray-code order, zero filter
//     slots for the classes a shift does not serve.  Measured before (14 MMAs of N = 16 .. 128 per K step, 98 per plane):
//     the kernel sat on the shared-memory A-operand feed, 4 KB per MMA whatever its N.
//   * for pad in {1, 2} the input shifts are 0 or +1 per axis (slab taps 1, 2; tap 0 is never used), so a slab carries one
//     halo line / column / plane on the high side only, and the ring is 3 deep (two live planes + one in flight).
//   * the issuer is one thread: the per-plane MMA list is the same for every plane and is built once as a table (descriptor
//     halves, instruction descriptor, accumulator column) -- with the group / chunk / K-step loops evaluated per plane the
//     kernel was bound by that thread's instruction stream.
//   * the epilogue may ACCUMULATE into the canvas (it holds the data gradient of conv_0_0 already: the sum of the two is what
//     the cost volume receives); old values are requested before the accumulator is waited for; 32-byte loads and stores.
constexpr int kKcMax = 3;
constexpr int kKcSlots = 3;
constexpr int kKcMaxMma = 8 * 7;       // MMAs per plane: 8 shifts x (112 / 16) K steps

struct DeconvKcParams {
    int B, Do, Ho, Wo;              // extent of the canvas that is written
    int Jd, Jh, Jw;                 // output lattice (voxel octets)
    int BW, L;                      // slab: BW voxels per line (the last one is halo), L output lines, BW * L <= 128
    int tiles_x, tiles_y;
    int dchunk, nchunks, n_items;
    int cout, n_rows;               // output channels, filter rows per tap in the packed weights
    int n_split;                    // CTAs that share an item, each NOUT output channels (blockIdx % n_split)
    int n_kc;                       // K chunks
    int kc_off[kKcMax], kc_n[kKcMax];   // first channel and channel count (16 / 32 / 64) of a chunk
    int kc_slab[kKcMax];            // byte offset of the chunk's sub-slab inside a ring slot
    int kc_w[kKcMax];               // byte offset of the chunk's filter region [n_slots][NOUT][kc_n] in shared memory
    int slab_bytes, w_bytes;        // ring slot, whole filter
    int accumulate;                 // 1: y += result
    int wide_io;                    // 1: 32-byte loads / stores (rows 32-byte aligned, channels in multiples of 16)
    int dbg;                        // diagnostics (MVSB200_KC_DBG): 1 = no MMAs, 2 = no slab loads, 8 = no stores
    DeconvWide g;
    long long y_sb, y_sd, y_sh, y_sw;
    __nv_bfloat16* y;
};

// K-major operand descriptor, row pitch (= swizzle span) given at run time: returns the high half; the low half is
// (addr >> 4) | 1 << 16
__device__ __forceinline__ uint32_t umma_desc_hi_rt(uint32_t rowb) {
    const uint32_t layout = rowb == 128 ? 2u : (rowb == 64 ? 4u : 6u);
    return ((8u * rowb) >> 4) | (1u << 14) | (layout << 29);       // SBO, descriptor version (bit 46), layout (bits 61..63)
}

__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

template <int NOUT>
__global__ void __launch_bounds__(kWgThreads, 1)
deconv3d_s2_kc_kernel(const __grid_constant__ CUtensorMap tm_x0, const __grid_constant__ CUtensorMap tm_x1,
                      const __grid_constant__ CUtensorMap tm_x2, const __grid_constant__ CUtensorMap tm_w0,
                      const __grid_constant__ CUtensorMap tm_w1, const __grid_constant__ CUtensorMap tm_w2,
                      const __grid_constant__ DeconvKcParams p) {
    // instruction descriptor without the N field: D fp32, A/B bf16, both K-major, M = 128; N = npos * NOUT per group
    constexpr uint32_t IDESC0 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
    constexpr uint32_t tmem_cols = 2 * 8 * NOUT;
    static_assert(NOUT == 16 || NOUT == 32, "accumulator columns");

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* w_smem = smem;
    unsigned char* slab_smem = smem + p.w_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(slab_smem + (size_t)kKcSlots * p.slab_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + kKcSlots;
    uint64_t* wfull = bars + 2 * kKcSlots;
    uint64_t* tfull = wfull + 1;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    uint4* mma_tab = reinterpret_cast<uint4*>(bars + 16);          // [2 * kKcMaxMma]: one entry per MMA of a plane (see the issuer)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.tiles_x * p.tiles_y;
    // this CTA's share of the output channels and its place among the CTAs that walk the items
    const int half = (int)blockIdx.x % p.n_split, walker = (int)blockIdx.x / p.n_split, n_walkers = (int)gridDim.x / p.n_split;
    const int row0 = half * NOUT;                        // first filter row == first output channel
    const int c_here = min(NOUT, p.cout - row0);

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x0) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w0) : "memory");
        for (int i = 0; i < kKcSlots; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        mbar_init(wfull, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    auto decode = [&](int item, int& b, int& d_begin, int& nd, int& x0, int& y0) {
        const int t = item % tiles, r = item / tiles;
        const int c = r % p.nchunks;
        b = r / p.nchunks;
        d_begin = c * p.dchunk;
        nd = min(p.dchunk, p.Jd - d_begin);
        x0 = (t % p.tiles_x) * (p.BW - 1);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            uint32_t wb = 0;
            for (int c = 0; c < p.n_kc; ++c) wb += (uint32_t)p.g.n_slots * NOUT * 2u * (uint32_t)p.kc_n[c];
            mbar_expect_tx(wfull, wb);
            for (int c = 0; c < p.n_kc; ++c) {
                const CUtensorMap* tm = c == 0 ? &tm_w0 : (c == 1 ? &tm_w1 : &tm_w2);
                const int tap_bytes = NOUT * 2 * p.kc_n[c];
                for (int e = 0; e < p.g.n_slots; ++e)      // tap 27 of the packed weights is all zeros
                    tma_load_2d(w_smem + p.kc_w[c] + e * tap_bytes, tm, wfull, 0, p.g.tap_k[e] * p.n_rows + row0);
            }
        }
        __syncwarp();
        uint32_t box_bytes = 0;
        for (int c = 0; c < p.n_kc; ++c) box_bytes += 2u * (uint32_t)p.kc_n[c] * p.BW * (p.L + 1);
        int gs = 0;
        for (int item = walker; item < p.n_items; item += n_walkers) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + 1; ++s, ++gs) {     // input planes d_begin + s
                const int slot = gs % kKcSlots;
                if (gs >= kKcSlots) mbar_wait(empty + slot, ((gs / kKcSlots) - 1) & 1);
                if (p.dbg & 2) { if (elect_one()) mbar_arrive(full + slot); }
                else if (elect_one()) {
                    mbar_expect_tx(full + slot, box_bytes);
                    for (int c = 0; c < p.n_kc; ++c) {
                        const CUtensorMap* tm = c == 0 ? &tm_x0 : (c == 1 ? &tm_x1 : &tm_x2);
                        tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes + p.kc_slab[c], tm, full + slot, p.kc_off[c], x0, y0,
                                    d_begin + s, b);
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        // The per-plane MMA list, built once in parallel by the lanes of this warp: entry = (A offset inside a ring slot |
        // depth shift, B descriptor low, descriptor high, instruction descriptor), (accumulator column | accumulate flag).
        const uint32_t w_base = (1u << 16) | (smem_u32(w_smem) >> 4);
        int n_mma = 0;
        {
            int per_group = 0;
            for (int c = 0; c < p.n_kc; ++c) per_group += p.kc_n[c] / 16;
            n_mma = p.g.n_groups * per_group;
            for (int e = lane; e < n_mma; e += 32) {
                const int g = e / per_group;
                int r = e - g * per_group, c = 0;
                while (r >= p.kc_n[c] / 16) { r -= p.kc_n[c] / 16; ++c; }
                const uint32_t rowb = 2u * (uint32_t)p.kc_n[c];
                const uint32_t rows = (uint32_t)((p.g.grp_th[g] - 1) * p.BW + (p.g.grp_tw[g] - 1));
                const uint32_t a_off = ((uint32_t)p.kc_slab[c] + rows * rowb + 32u * (uint32_t)r) >> 4;
                const uint32_t b_lo = w_base + (((uint32_t)p.kc_w[c] + (uint32_t)p.g.grp_slot0[g] * NOUT * rowb + 32u * (uint32_t)r) >> 4);
                const uint32_t acc = (p.g.grp_first[g] && c == 0 && r == 0) ? 0u : 1u;
                mma_tab[2 * e] = make_uint4(a_off | (p.g.grp_td[g] == 2 ? 0x80000000u : 0u), b_lo, umma_desc_hi_rt(rowb),
                                            IDESC0 | ((uint32_t)((p.g.grp_npos[g] * NOUT) >> 3) << 17));
                mma_tab[2 * e + 1] = make_uint4((uint32_t)(p.g.grp_pos0[g] * NOUT) | (acc << 16), 0u, 0u, 0u);
            }
            __syncwarp();
        }
        mbar_wait(wfull, 0);
        const uint32_t slab_base = (1u << 16) | (smem_u32(slab_smem) >> 4);
        const uint32_t slab16 = (uint32_t)p.slab_bytes >> 4;
        int gs0 = 0, gp = 0, landed = 0;
        for (int item = walker; item < p.n_items; item += n_walkers) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                if (gp >= 2) mbar_wait(tempty + stage, ((gp >> 1) - 1) & 1);
                while (landed <= gs0 + d + 1) { mbar_wait(full + landed % kKcSlots, (landed / kKcSlots) & 1); ++landed; }
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t slot_lo0 = slab_base + (uint32_t)((gs0 + d) % kKcSlots) * slab16;
                    const uint32_t slot_lo1 = slab_base + (uint32_t)((gs0 + d + 1) % kKcSlots) * slab16;
                    const uint32_t t_stage = tmem_base + (uint32_t)(stage * 8 * NOUT);
#pragma unroll 4
                    for (int e = 0; e < ((p.dbg & 1) ? 0 : n_mma); ++e) {
                        const uint4 u = mma_tab[2 * e];
                        const uint32_t v = mma_tab[2 * e + 1].x;
                        const uint32_t a_lo = (u.x & 0x7fffffffu) + ((u.x >> 31) ? slot_lo1 : slot_lo0);
                        umma_bf16_lohi(t_stage + (v & 0xffffu), a_lo, u.z, u.y, u.z, u.w, v >> 16);
                    }
                    umma_commit(empty + (gs0 + d) % kKcSlots);
                    if (d == nd - 1) umma_commit(empty + (gs0 + nd) % kKcSlots);
                    umma_commit(tfull + stage);
                }
                __syncwarp();
            }
            gs0 += nd + 1;
        }
    } else {
        // ===================================== epilogue =========================================
        const int q = warp & 3;
        const int m = q * 32 + lane;
        const int tj = m / p.BW, ti = m - tj * p.BW;
        const bool in_tile = ti < p.BW - 1 && tj < p.L;
        int cls[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) cls[c] = p.g.cls_of_pos[c];
        int gp = 0;
        for (int item = walker; item < p.n_items; item += n_walkers) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            const int ox = 2 * (x0 + ti), oy = 2 * (y0 + tj);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                const int oz = 2 * (d_begin + d);
                __nv_bfloat16* base = p.y + (long long)b * p.y_sb + (long long)oz * p.y_sd + (long long)oy * p.y_sh + (long long)ox * p.y_sw + row0;
                U8 old[8][NOUT / 16];
                bool ok[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int pd = cls[c] >> 2, ph = cls[c] >> 1 & 1, pw = cls[c] & 1;
                    ok[c] = in_tile && oz + pd < p.Do && oy + ph < p.Ho && ox + pw < p.Wo;
                    if (p.accumulate && ok[c]) {
                        const __nv_bfloat16* row = base + pd * p.y_sd + ph * p.y_sh + pw * p.y_sw;
#pragma unroll
                        for (int j = 0; j < NOUT / 16; ++j) {
                            if (p.wide_io) {
                                if (j * 16 < c_here) old[c][j] = ld_u8(row + 16 * j);
                            } else {
#pragma unroll
                                for (int h = 0; h < 2; ++h)
                                    if (j * 16 + 8 * h < c_here) {
                                        const uint4 t = *reinterpret_cast<const uint4*>(row + 16 * j + 8 * h);
                                        old[c][j].v[4 * h] = t.x; old[c][j].v[4 * h + 1] = t.y; old[c][j].v[4 * h + 2] = t.z; old[c][j].v[4 * h + 3] = t.w;
                                    }
                            }
                        }
                    }
                }
                mbar_wait(tfull + stage, (gp >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    uint32_t v[NOUT];
                    tmem_ld<NOUT>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((stage * 8 + c) * NOUT), v);
                    tmem_ld_wait();
                    if (ok[c] && !(p.dbg & 8)) {
                        const int pd = cls[c] >> 2, ph = cls[c] >> 1 & 1, pw = cls[c] & 1;
                        __nv_bfloat16* row = base + pd * p.y_sd + ph * p.y_sh + pw * p.y_sw;
#pragma unroll
                        for (int j = 0; j < NOUT / 16; ++j) {
                            if (j * 16 < c_here) {
                                U8 o;
#pragma unroll
                                for (int i = 0; i < 8; ++i) {
                                    float lo = __uint_as_float(v[j * 16 + 2 * i]), hi = __uint_as_float(v[j * 16 + 2 * i + 1]);
                                    if (p.accumulate) { lo += bf16_lo(old[c][j].v[i]); hi += bf16_hi(old[c][j].v[i]); }
                                    o.v[i] = pack_bf16x2(lo, hi);
                                }
                                if (p.wide_io) st_u8(row + 16 * j, o);
                                else {
#pragma unroll
                                    for (int h = 0; h < 2; ++h)
                                        if (j * 16 + 8 * h < c_here)
                                            *reinterpret_cast<uint4*>(row + 16 * j + 8 * h) = make_uint4(o.v[4 * h], o.v[4 * h + 1], o.v[4 * h + 2], o.v[4 * h + 3]);
                                }
                            }
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(tempty + stage);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

template <int NOUT>
int launch_deconv_kc(const void* x, int x_cs, const void* w, const int* kc_off, const int* kc_n, int n_kc, void* y, int B, int Di,
                     int Hi, int Wi, int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                     const long long* ys, int accumulate, cudaStream_t st) {
    DeconvKcParams p;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo;
    p.Jd = (Do + 1) / 2; p.Jh = (Ho + 1) / 2; p.Jw = (Wo + 1) / 2;
    p.cout = cout; p.n_rows = n_rows; p.n_kc = n_kc; p.accumulate = accumulate;
    p.n_split = (cout + NOUT - 1) / NOUT;
    p.dbg = 0;
    if (const char* e = getenv("MVSB200_KC_DBG")) p.dbg = atoi(e);
    MVS_TRY(build_deconv_wide(pad_d, pad_h, pad_w, NOUT, p.g));
    {
        int ksteps = 0;
        for (int c = 0; c < n_kc; ++c) ksteps += kc_n[c] / 16;
        MVS_REQUIRE(p.g.n_groups * ksteps <= kKcMaxMma, "deconv3d_s2_kc: %d MMAs per plane exceed the table", p.g.n_groups * ksteps);
    }
    // filter regions
    int woff = 0;
    for (int c = 0; c < kKcMax; ++c) {
        p.kc_off[c] = c < n_kc ? kc_off[c] : 0;
        p.kc_n[c] = c < n_kc ? kc_n[c] : 0;
        p.kc_w[c] = woff;
        if (c < n_kc) woff += (p.g.n_slots * NOUT * 2 * kc_n[c] + 1023) / 1024 * 1024;
    }
    p.w_bytes = woff;
    // slab geometry: BW * L <= 128 rows, one halo column / line
    const size_t budget = 227 * 1024 - 1024 - 128 - 32 * kKcMaxMma;
    double best = -1.0;
    for (int BW = 3; BW <= 128; ++BW) {
        const int L = 128 / BW;
        if (L < 1 || L + 1 > 256) continue;
        const int rows = 128 + BW + 2;
        size_t slab = 0;
        for (int c = 0; c < n_kc; ++c) slab += ((size_t)rows * 2 * kc_n[c] + 1023) / 1024 * 1024;
        if ((size_t)p.w_bytes + kKcSlots * slab > budget) continue;
        const int tx = (p.Jw + BW - 2) / (BW - 1), ty = (p.Jh + L - 1) / L;
        const double eff = (double)p.Jw * p.Jh / ((double)tx * ty * 128);
        if (eff > best) { best = eff; p.BW = BW; p.L = L; p.tiles_x = tx; p.tiles_y = ty; p.slab_bytes = (int)slab; }
    }
    MVS_REQUIRE(best > 0, "deconv3d_s2_kc: no slab geometry fits shared memory (%d K chunks, N=%d)", n_kc, NOUT);
    {
        const int rows = 128 + p.BW + 2;
        int off = 0;
        for (int c = 0; c < kKcMax; ++c) {
            p.kc_slab[c] = off;
            if (c < n_kc) off += (rows * 2 * kc_n[c] + 1023) / 1024 * 1024;
        }
    }
    CUtensorMap tm_x[kKcMax], tm_w[kKcMax];
    const char* wp = reinterpret_cast<const char*>(w);
    for (int c = 0; c < n_kc; ++c) {
        MVS_TRY(encode_volume(&tm_x[c], x, x_cs, kc_n[c], Wi, Hi, Di, B, p.BW, p.L + 1, "deconv3d_s2_kc", "x, chunk", c));
        // packed filter of the chunk: [28 * n_rows][kc_n] bf16 (tap 27 = zeros), chunks one after the other
        MVS_TRY(encode_filter(&tm_w[c], wp, kc_n[c], 28 * n_rows, NOUT, "deconv3d_s2_kc", "w, chunk", c));
        wp += (size_t)28 * n_rows * 2 * kc_n[c];
    }
    for (int c = n_kc; c < kKcMax; ++c) { tm_x[c] = tm_x[0]; tm_w[c] = tm_w[0]; }
    p.y_sb = ys[0]; p.y_sd = ys[1]; p.y_sh = ys[2]; p.y_sw = ys[3];
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.wide_io = (cout % 16 == 0 && ys[0] % 16 == 0 && ys[1] % 16 == 0 && ys[2] % 16 == 0 && ys[3] % 16 == 0 && ((uintptr_t)y & 31u) == 0) ? 1 : 0;
    const long tiles = (long)p.tiles_x * p.tiles_y;
    const int sms = sm_count();
    const long walkers_max = sms / p.n_split > 0 ? sms / p.n_split : 1;
    const Runs runs = choose_runs(tiles, B, p.Jd, walkers_max, 3);
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    p.n_items = (int)(tiles * p.nchunks * B);
    const long walkers = p.n_items < walkers_max ? p.n_items : walkers_max;
    if (p.dbg & 4) fprintf(stderr, "kc: NOUT=%d split=%d BW=%d L=%d tiles=%dx%d dchunk=%d nchunks=%d items=%d groups=%d slots=%d slab=%d w=%d\n", NOUT, p.n_split, p.BW, p.L, p.tiles_x, p.tiles_y, p.dchunk, p.nchunks, p.n_items, p.g.n_groups, p.g.n_slots, p.slab_bytes, p.w_bytes);
    const dim3 grid((unsigned)(walkers * p.n_split), 1, 1);
    const size_t smem = 1024 + (size_t)p.w_bytes + (size_t)kKcSlots * p.slab_bytes + 128 + 32 * kKcMaxMma;
    MVS_CUDA(cudaFuncSetAttribute(deconv3d_s2_kc_kernel<NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    deconv3d_s2_kc_kernel<NOUT><<<grid, kWgThreads, smem, st>>>(tm_x[0], tm_x[1], tm_x[2], tm_w[0], tm_w[1], tm_w[2], p);
    MVS_CHECK_LAUNCH("deconv3d_s2_kc");
    return MVSB200_OK;
}

}  // namespace

/* Weight gradient of the stride-2 layers, one launch (see the header of this file):
 *   gw[k][cb][cs] = sum_o big(2o - pad + k)[cb] * small(o)[cs]. */
extern "C" int mvsb200_conv3d_s2_wgrad_lines(const void* big, const void* small, float* gw, int B, int Db, int Hb, int Wb, int Cb,
                                             int Ds, int Hs, int Ws, int Cs, int pad_d, int pad_h, int pad_w,
                                             const int64_t* small_strides4, void* stream) {
    const char* name = "conv3d_s2_wgrad_lines";
    MVS_TRY(check_pointers(name, {big, small, gw}));
    MVS_REQUIRE(B >= 1 && B <= 65535 && Db >= 1 && Hb >= 1 && Wb >= 2 && Ds >= 1 && Hs >= 1 && Ws >= 1, "%s: bad shape", name);
    MVS_REQUIRE(Wb % 2 == 0, "%s: the strided operand needs an even number of voxels per line (got %d)", name, Wb);
    MVS_REQUIRE(Ws + 1 <= 256, "%s: lines of the dense operand are limited to 255 voxels (got %d)", name, Ws);
    MVS_REQUIRE(Cb == 8 || Cb == 16 || Cb == 32, "%s: the strided operand must have 8, 16 or 32 channels (got %d)", name, Cb);
    MVS_REQUIRE(Cs == 16 || Cs == 32 || Cs == 64 || (Cs > 64 && Cs <= 128 && Cs % 16 == 0),
                "%s: the dense operand needs 16, 32, 64 or 80..128 (multiple of 16) channels (got %d)", name, Cs);
    MVS_TRY(check_pads(name, pad_d, pad_h, pad_w));
    long long ssv[4];
    const long long* ss = nullptr;
    if (small_strides4) {
        for (int i = 0; i < 4; ++i) {
            ssv[i] = (long long)small_strides4[i];
            MVS_REQUIRE(ssv[i] > 0 && ssv[i] % 8 == 0, "%s: strides of the dense operand must be positive multiples of 8 elements", name);
        }
        ss = ssv;
    }
    cudaStream_t st = (cudaStream_t)stream;
    MVS_CUDA(cudaMemsetAsync(gw, 0, (size_t)27 * Cb * Cs * sizeof(float), st));
    if (Cb == 8) return launch_s2_wgrad_lines<8>(big, small, gw, B, Db, Hb, Wb, Ds, Hs, Ws, Cs, pad_d, pad_h, pad_w, ss, st);
    if (Cb == 16) return launch_s2_wgrad_lines<16>(big, small, gw, B, Db, Hb, Wb, Ds, Hs, Ws, Cs, pad_d, pad_h, pad_w, ss, st);
    return launch_s2_wgrad_lines<32>(big, small, gw, B, Db, Hb, Wb, Ds, Hs, Ws, Cs, pad_d, pad_h, pad_w, ss, st);
}

/* Stride-2 TRANSPOSED convolution whose input channels come in K CHUNKS of 16 / 32 / 64 (deconv3d_s2_kc_kernel): the data
 * gradient of the stacked branches conv_{1,2,3}_0 (112 -> 32).  See the header of the kernel. */
extern "C" int mvsb200_deconv3d_s2_kc_fwd(const void* x, int x_cs, const void* w_packed, const int* kc_off, const int* kc_n, int n_kc,
                                          void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout, int n_rows,
                                          int pad_d, int pad_h, int pad_w, const int64_t* y_strides4, int accumulate, void* stream) {
    const char* name = "deconv3d_s2_kc_fwd";
    MVS_TRY(check_pointers(name, {x, w_packed, y}, {y_strides4, kc_off, kc_n}));
    MVS_REQUIRE(B >= 1 && B <= 65535 && Di >= 1 && Hi >= 1 && Wi >= 1 && Do >= 1 && Ho >= 1 && Wo >= 1, "%s: bad shape", name);
    MVS_REQUIRE(n_kc >= 1 && n_kc <= 3 && x_cs % 8 == 0, "%s: 1..3 K chunks, channel stride a multiple of 8 (got %d, %d)", name, n_kc, x_cs);
    int ktot = 0;
    for (int c = 0; c < n_kc; ++c) {
        MVS_REQUIRE(kc_n[c] == 16 || kc_n[c] == 32 || kc_n[c] == 64, "%s: a K chunk has 16, 32 or 64 channels (got %d)", name, kc_n[c]);
        MVS_REQUIRE(kc_off[c] >= 0 && kc_off[c] % 8 == 0 && kc_off[c] + kc_n[c] <= x_cs, "%s: K chunk %d outside the voxel row", name, c);
        ktot += kc_n[c];
    }
    MVS_REQUIRE(cout >= 8 && cout % 8 == 0 && cout <= n_rows && n_rows % 16 == 0 && n_rows <= 64,
                "%s: cout must be a multiple of 8 and n_rows a multiple of 16 <= 64 (cout=%d n_rows=%d)", name, cout, n_rows);
    MVS_TRY(check_pads(name, pad_d, pad_h, pad_w));
    long long ys[4];
    MVS_TRY(copy_strides(name, y_strides4, ys));
    cudaStream_t st = (cudaStream_t)stream;
    // output channels per CTA: 32 while the filter (31 slots x 32 x K) and three slabs fit shared memory, else 16; the CTAs of
    // one launch share the channel groups (blockIdx % n_split)
    const int nout = ktot <= 64 && n_rows % 32 == 0 ? 32 : 16;
    const int rc = nout == 32
        ? launch_deconv_kc<32>(x, x_cs, w_packed, kc_off, kc_n, n_kc, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, n_rows, pad_d, pad_h, pad_w, ys, accumulate, st)
        : launch_deconv_kc<16>(x, x_cs, w_packed, kc_off, kc_n, n_kc, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, n_rows, pad_d, pad_h, pad_w, ys, accumulate, st);
    if (rc != MVSB200_OK) return rc;
    return MVSB200_OK;
}
