// K3: 3x3x3 stride-1 convolution of channel-last bf16 volumes as an implicit GEMM on tcgen05 tensor cores (sm_100a).
//
// Reference semantics (citations into /root/reference/scripts):
//   model.py:223-234   Conv3d(k=3, stride, padding, bias=False)  -- the stride-1 layers conv_0_0, conv_{1,2,3}_1
//   model.py:101-113   their use in CostVolumeReg.forward; autograd's dgrad of the same layers is this very
//                      convolution with the flipped, transposed filter (host side packs it)
//
// GEMM view: D[M = voxels, N = Cout] += A[M, K = Cin] * B[K, N] summed over the 27 taps.  The design removes the
// 27-fold re-read of the activations that a tap-by-tap im2col costs:
//   * a CTA owns an (x, y) tile of the volume and MARCHES ALONG DEPTH.  Per input plane ONE TMA tile load brings the
//     (L+2) x BW halo'd slab of voxel rows (Cin bf16 each, hardware-swizzled) into a 4-slot shared-memory ring; every
//     slab is used by the three output planes around it.
//   * inside a slab the 9 in-plane taps are NOT separate copies: voxel rows are consecutive in shared memory, so the
//     A operand of tap (kh, kw) is the same slab read from row offset kh*BW + kw -- only the start address of the
//     UMMA shared-memory descriptor changes.  Output rows that fall on the halo columns are computed and dropped
//     (BW-2 useful of BW).
//   * all 27 x Cout x Cin filter taps stay resident in shared memory (loaded once per CTA by TMA).
//   * accumulators live in TMEM (MB blocks of 128 rows x NOUT fp32 columns, double buffered), the epilogue warps read
//     them back with tcgen05.ld, convert to bf16 and store voxel rows while the MMA warp works on the next plane.
// Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane) + TMEM allocator, warps 2..5 = epilogue.
#include "tc_common.cuh"
#include <stdlib.h>
#include <type_traits>

using namespace mvsb200;

namespace {

constexpr int kTcThreads = 192;
constexpr int kSlots3 = 4;          // slab ring depth (3 live planes + 1 in flight)
constexpr int kMaxMB = 4;

struct ConvParams {
    int B, Do, Ho, Wo;              // output volume
    int off_d, off_h, off_w;        // input coordinate = output coordinate + tap + off   (-1 = padding 1, 0 = valid)
    int BW, L, MB;                  // slab: BW voxels per line (incl. 2 halo), L output lines, MB 128-row blocks
    int tiles_x, tiles_y;
    int dchunk, nchunks;            // output planes per item, depth runs per volume
    int n_items;                    // B * nchunks * tiles_x * tiles_y work items
    int cout, y_cs, y_coff;         // channels to store, channel stride of an output voxel row, first channel
    int n_rows;                     // filter rows per tap in the packed weights (multiple of 16)
    int w_row0;                     // first filter row this launch computes (N split of wide layers)
    int slab_bytes;                 // per ring slot, multiple of 1024
    unsigned tap_mask;              // bit (kd*3+kh)*3+kw: tap present (absent taps are neither loaded nor multiplied)
    long long y_sb, y_sd, y_sh, y_sw;   // output voxel-row strides in elements (a parity sub-lattice of a canvas, or dense)
    __nv_bfloat16* y;
};


// Persistent kernel: CTA c works on items c, c + gridDim.x, ...; an item is (batch, depth run, xy tile).  The filter is
// loaded once per CTA; the slab ring, the TMEM stages and all mbarrier phases run on across items (global counters).
template <int CIN, int NOUT>
__global__ void __launch_bounds__(kTcThreads, 1)
conv3d_s1_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w, const ConvParams p) {
    constexpr int ROWB = CIN * 2;                       // bytes per voxel row == swizzle span
    constexpr int KSTEPS = CIN / 16;                    // UMMA K = 16 bf16 = 32 bytes
    constexpr int W_TAP_BYTES = NOUT * ROWB;
    constexpr int W_BYTES = 27 * W_TAP_BYTES;
    constexpr int W_BYTES_AL = (W_BYTES + 1023) / 1024 * 1024;
    // instruction descriptor: D fp32, A/B bf16, both K-major, N, M = 128
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NOUT >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* w_smem = smem;
    unsigned char* slab_smem = smem + W_BYTES_AL;
    uint64_t* bars = reinterpret_cast<uint64_t*>(slab_smem + (size_t)kSlots3 * p.slab_bytes);
    uint64_t* full = bars;                  // [kSlots3]  slab landed
    uint64_t* empty = bars + kSlots3;       // [kSlots3]  slab no longer read by any MMA
    uint64_t* wfull = bars + 2 * kSlots3;   // [1]        filter resident
    uint64_t* tfull = wfull + 1;            // [2]        accumulator stage complete
    uint64_t* tempty = tfull + 2;           // [2]        accumulator stage drained by the epilogue
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int MB = p.MB;
    const int tiles = p.tiles_x * p.tiles_y;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * MB * NOUT) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w) : "memory");
        for (int i = 0; i < kSlots3; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
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

    // item -> (b, d_begin, nd, x0, y0)
    auto decode = [&](int item, int& b, int& d_begin, int& nd, int& x0, int& y0) {
        const int t = item % tiles, r = item / tiles;
        const int c = r % p.nchunks;
        b = r / p.nchunks;
        d_begin = c * p.dchunk;
        nd = min(p.dchunk, p.Do - d_begin);
        x0 = (t % p.tiles_x) * (p.BW - 2);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            mbar_expect_tx(wfull, (uint32_t)__popc(p.tap_mask) * W_TAP_BYTES);
            for (int tap = 0; tap < 27; ++tap)
                if (p.tap_mask >> tap & 1u) tma_load_2d(w_smem + tap * W_TAP_BYTES, &tm_w, wfull, 0, tap * p.n_rows + p.w_row0);
        }
        __syncwarp();
        const uint32_t box_bytes = (uint32_t)ROWB * p.BW * (p.L + 2);
        int gs = 0;                                      // slabs loaded so far (all items)
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + 2; ++s, ++gs) {     // input planes d_begin+off_d+s
                const int slot = gs % kSlots3;
                if (gs >= kSlots3) mbar_wait(empty + slot, ((gs / kSlots3) - 1) & 1);
                if (elect_one()) {
                    mbar_expect_tx(full + slot, box_bytes);
                    tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, &tm_x, full + slot, 0, x0 + p.off_w, y0 + p.off_h,
                                d_begin + p.off_d + s, b);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        mbar_wait(wfull, 0);
        const uint64_t d0 = umma_desc<ROWB>(0);
        const uint32_t desc_hi = (uint32_t)(d0 >> 32);
        const uint32_t w_lo = (uint32_t)d0 | (smem_u32(w_smem) >> 4);
        const uint32_t slab_lo = (uint32_t)d0 | (smem_u32(slab_smem) >> 4);
        const uint32_t bw16 = (uint32_t)(p.BW * ROWB) >> 4, slab16 = (uint32_t)p.slab_bytes >> 4;
        int gs0 = 0, gp = 0, landed = 0;                 // first slab of the item, planes issued, slabs waited for
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                if (gp >= 2) mbar_wait(tempty + stage, ((gp >> 1) - 1) & 1);
                while (landed <= gs0 + d + 2) { mbar_wait(full + landed % kSlots3, (landed / kSlots3) & 1); ++landed; }
                tc_fence_after();
                if (elect_one()) {
                    uint32_t slot_lo[3];
#pragma unroll
                    for (int kd = 0; kd < 3; ++kd) slot_lo[kd] = slab_lo + (uint32_t)((gs0 + d + kd) % kSlots3) * slab16;
                    for (int mb = 0; mb < MB; ++mb) {
                        const uint32_t d_tmem = tmem_base + (uint32_t)((stage * MB + mb) * NOUT);
                        const uint32_t mb16 = (uint32_t)(mb * 128 * ROWB) >> 4;
                        uint32_t acc = 0;
#pragma unroll
                        for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
                            for (int kh = 0; kh < 3; ++kh) {
                                const uint32_t row_lo = slot_lo[kd] + mb16 + kh * bw16;
#pragma unroll
                                for (int kw = 0; kw < 3; ++kw) {
                                    if (p.tap_mask >> ((kd * 3 + kh) * 3 + kw) & 1u) {
#pragma unroll
                                        for (int k = 0; k < KSTEPS; ++k) {
                                            umma_bf16_lohi(d_tmem, row_lo + (uint32_t)((kw * ROWB + k * 32) >> 4), desc_hi,
                                                           w_lo + (uint32_t)((((kd * 3 + kh) * 3 + kw) * W_TAP_BYTES + k * 32) >> 4),
                                                           desc_hi, IDESC, acc);
                                            acc = 1;
                                        }
                                    }
                                }
                            }
                        }
                    }
                    umma_commit(empty + (gs0 + d) % kSlots3);      // input plane s = d is not read after this output plane
                    if (d == nd - 1) {                               // end of the run: its two trailing halo planes too
                        umma_commit(empty + (gs0 + nd) % kSlots3);
                        umma_commit(empty + (gs0 + nd + 1) % kSlots3);
                    }
                    umma_commit(tfull + stage);
                }
                __syncwarp();
            }
            gs0 += nd + 2;
        }
    } else {
        // ===================================== epilogue =========================================
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        int rel[kMaxMB], ti[kMaxMB], tj[kMaxMB];          // this thread's row of each 128-row block inside the tile
#pragma unroll
        for (int mb = 0; mb < kMaxMB; ++mb) {
            const int m = mb * 128 + q * 32 + lane;
            tj[mb] = m / p.BW; ti[mb] = m - tj[mb] * p.BW;
            rel[mb] = (ti[mb] < p.BW - 2 && tj[mb] < p.L) ? 1 : -1;
        }
        int gp = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                mbar_wait(tfull + stage, (gp >> 1) & 1);
                tc_fence_after();
                __nv_bfloat16* plane0 = p.y + (long long)b * p.y_sb + (long long)(d_begin + d) * p.y_sd + (long long)y0 * p.y_sh + (long long)x0 * p.y_sw + p.y_coff;
#pragma unroll
                for (int mb = 0; mb < kMaxMB; ++mb) {
                    if (mb < MB) {
                        uint32_t v[NOUT];
                        tmem_ld<NOUT>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((stage * MB + mb) * NOUT), v);
                        tmem_ld_wait();
                        if (rel[mb] >= 0 && x0 + ti[mb] < p.Wo && y0 + tj[mb] < p.Ho) {
                            __nv_bfloat16* row = plane0 + (long long)tj[mb] * p.y_sh + (long long)ti[mb] * p.y_sw;
#pragma unroll
                            for (int c = 0; c < NOUT; c += 8) {
                                if (c < p.cout) {
                                    const uint4 o = make_uint4(pack_bf16x2(__uint_as_float(v[c]), __uint_as_float(v[c + 1])),
                                                               pack_bf16x2(__uint_as_float(v[c + 2]), __uint_as_float(v[c + 3])),
                                                               pack_bf16x2(__uint_as_float(v[c + 4]), __uint_as_float(v[c + 5])),
                                                               pack_bf16x2(__uint_as_float(v[c + 6]), __uint_as_float(v[c + 7])));
                                    *reinterpret_cast<uint4*>(row + c) = o;
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


struct TilePlan {
    int BW, L, MB, tiles_x, tiles_y, slab_bytes;
    double score;
};

// Slab geometry for MB 128-row blocks: BW voxels per line of which `halo` are halo columns, L = MB * 128 / BW output lines
// plus `halo` halo lines, `slots` slabs in the ring next to the resident filter.  Maximises useful rows per MMA row and per
// loaded row over BW = bw0, bw0 + bw_step, ... 256 within the shared-memory budget; the first BW wins a tie.  score <= 0:
// nothing fits.
TilePlan plan_slab(int Ho, int Wo, int rowb, size_t w_bytes_al, size_t smem_budget, int MB, int slots, int halo, int bw0,
                   int bw_step) {
    TilePlan best{};
    best.score = -1.0;
    for (int BW = bw0; BW <= 256; BW += bw_step) {
        const int L = (MB * 128) / BW;
        if (L < 1 || L + halo > 256) continue;
        const int rows = MB * 128 + halo * BW + 2;
        const int slab = ((rows * rowb) + 1023) / 1024 * 1024;
        if (w_bytes_al + (size_t)slots * slab + 256 > smem_budget) continue;
        const int tiles_x = (Wo + BW - 1 - halo) / (BW - halo), tiles_y = (Ho + L - 1) / L;
        const double mma_eff = (double)Wo * Ho / ((double)tiles_x * tiles_y * MB * 128);
        const double load_eff = (double)Wo * Ho / ((double)tiles_x * tiles_y * (L + halo) * BW);
        const double score = mma_eff * (0.5 + 0.5 * load_eff);
        if (score > best.score) best = TilePlan{BW, L, MB, tiles_x, tiles_y, slab, score};
    }
    return best;
}

// the best slab over MB = 1, 2, 4 blocks (the smaller MB wins a tie)
TilePlan plan_tiles(int Ho, int Wo, int rowb, size_t w_bytes_al, size_t smem_budget, int slots, int halo, int bw0, int bw_step) {
    TilePlan best{};
    best.score = -1.0;
    for (int MB = 1; MB <= kMaxMB; MB *= 2) {
        const TilePlan tp = plan_slab(Ho, Wo, rowb, w_bytes_al, smem_budget, MB, slots, halo, bw0, bw_step);
        if (tp.score > best.score) best = tp;
    }
    return best;
}

template <int CIN, int NOUT>
int launch_conv(const void* x, const void* w, void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout,
                int y_cs, int y_coff, int n_rows, int w_row0, int off_d, int off_h, int off_w, unsigned tap_mask,
                const long long* y_strides4, cudaStream_t st) {
    constexpr int ROWB = CIN * 2;
    constexpr size_t W_BYTES_AL = ((size_t)27 * NOUT * ROWB + 1023) / 1024 * 1024;
    const size_t smem_budget = 227 * 1024 - 1024;       // 1024 for the manual alignment of the dynamic window
    const TilePlan tp = plan_tiles(Ho, Wo, ROWB, W_BYTES_AL, smem_budget, kSlots3, 2, 10, 2);
    MVS_REQUIRE(tp.score > 0, "conv3d_s1: no slab geometry fits shared memory (Cin=%d, N=%d)", CIN, NOUT);

    CUtensorMap tm_x, tm_w;
    MVS_TRY(encode_volume(&tm_x, x, CIN, CIN, Wi, Hi, Di, B, tp.BW, tp.L + 2, "conv3d_s1", "x"));
    MVS_TRY(encode_filter(&tm_w, w, CIN, 27 * n_rows, NOUT, "conv3d_s1", "w"));

    ConvParams p;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo;
    p.off_d = off_d; p.off_h = off_h; p.off_w = off_w;
    p.BW = tp.BW; p.L = tp.L; p.MB = tp.MB; p.tiles_x = tp.tiles_x; p.tiles_y = tp.tiles_y;
    p.cout = cout; p.y_cs = y_cs; p.y_coff = y_coff; p.n_rows = n_rows; p.w_row0 = w_row0;
    p.slab_bytes = tp.slab_bytes;
    p.tap_mask = tap_mask & 0x7ffffffu;
    if (y_strides4) {
        p.y_sb = y_strides4[0]; p.y_sd = y_strides4[1]; p.y_sh = y_strides4[2]; p.y_sw = y_strides4[3];
    } else {
        p.y_sw = y_cs; p.y_sh = (long long)Wo * y_cs; p.y_sd = (long long)Ho * Wo * y_cs; p.y_sb = (long long)Do * Ho * Wo * y_cs;
    }
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    // depth runs: an item costs its planes + 2 halo planes + ~2 planes of pipeline fill; one persistent CTA per SM
    const long tiles = (long)tp.tiles_x * tp.tiles_y;
    const int sms = sm_count();
    const Runs runs = choose_runs(tiles, B, Do, sms, 4);
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    if (const char* e = getenv("MVSB200_CONV_DCHUNK")) {
        int v = atoi(e);
        if (v > 0) { p.dchunk = v < Do ? v : Do; p.nchunks = (Do + p.dchunk - 1) / p.dchunk; }
    }
    p.n_items = (int)(tiles * p.nchunks * B);
    const dim3 grid((unsigned)(p.n_items < sms ? p.n_items : sms), 1, 1);
    const size_t smem = 1024 + W_BYTES_AL + (size_t)kSlots3 * tp.slab_bytes + 256;
    MVS_CUDA(cudaFuncSetAttribute(conv3d_s1_tc_kernel<CIN, NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv3d_s1_tc_kernel<CIN, NOUT><<<grid, kTcThreads, smem, st>>>(tm_x, tm_w, p);
    MVS_CHECK_LAUNCH("conv3d_s1_tc");
    return MVSB200_OK;
}

// =================================================================================================================
// Weight gradient of the same convolution on tcgen05:  gW[tap][ci][co] = sum_v x(v + tap + off)[ci] * gy(v)[co].
// The REDUCTION runs over voxels: D[M, N] += A[M, K = 16 voxels] * B[K, N].  In shared memory both operands have the voxel
// (K) as the row and the channels contiguous, i.e. they are MN-major UMMA operands, and a swizzle atom of an MN-major
// operand may start at ANY row -- which lets one MMA cover 9 taps of a depth slice:
//   A = the halo'd, TMA-written x slab of the forward kernel.  Its M extent is built from atoms of Cin channels whose
//       stride (the descriptor's leading byte offset) is ONE VOXEL ROW: atom kw is the slab shifted by kw voxels, so
//       D rows are (kw, ci).
//   B = the gy tile of the plane, written by TMA line by line at the slab's pitch BW behind 2*BW rows of zeros (halo
//       columns and everything outside the tile stay zero).  Its N extent is built from atoms of co channels whose
//       stride is ONE LINE (BW rows): atom n is the tile shifted by n lines, so D columns are (kh = 2 - n, co):
//       sum_v x[v + kw] * gy[v - kh*BW] = sum_r x[r + kh*BW + kw] * gy[r].
// One accumulator block per depth tap kd stays in TMEM over the CTA's whole run (<= 512 columns; 64-channel gy in
// 32-channel halves, 64-channel x with its third kw tap in a second block) and is added to gW with fp32 reductions.
struct WgradParams {
    int B, Do, Ho, Wo;              // gy volume
    int off_d, off_h, off_w;
    int BW, L;                      // slab pitch (voxels per line incl. 2 halo), gy lines per tile
    int tiles_x, tiles_y;
    int dchunk, nchunks, n_items;
    int n_roles;                    // (gy channel chunk, depth taps) combinations shared out over the CTAs (blockIdx % n_roles)
    int role_co0[8];                // first gy channel of a role
    int role_kd[8];                 // depth taps of a role (bit kd); the others' MMAs are not issued
    int cout;                       // real output channels of the layer (row length of gW)
    int slab_bytes, gy_bytes;       // per ring slot / per gy stage, multiples of 1024
    int ksteps;                     // ceil((L+2)*BW / 16)
    int tap_map[27];                // kernel tap (kd*3+kh)*3+kw -> row block of gw it is added to, -1 = dropped
    float* gw;                      // [27][CIN][cout] fp32, accumulated into
};


template <int CIN, int NCO>
__global__ void __launch_bounds__(kTcThreads, 1)
conv3d_s1_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_g, const WgradParams p) {
    constexpr int ROWX = CIN * 2, ROWG = NCO * 2;
    constexpr int UN = (3 * NCO + 15) / 16 * 16;        // UMMA N: atoms kh = 2,1,0 (+ a junk atom when 3*NCO % 16 != 0)
    constexpr int KWB = CIN == 64 ? 2 : 1;              // A blocks per depth tap: 64-channel atoms fit twice into M = 128
    // D fp32, A/B bf16, A and B MN-major, N = UN, M = 128
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(UN >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* slab_smem = smem;
    unsigned char* gy_smem = smem + (size_t)kSlots3 * p.slab_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(gy_smem + (size_t)2 * p.gy_bytes);
    uint64_t* full = bars;                  // [kSlots3] x slab landed
    uint64_t* empty = bars + kSlots3;       // [kSlots3] x slab free
    uint64_t* gfull = bars + 2 * kSlots3;   // [2] gy tile landed
    uint64_t* gempty = gfull + 2;           // [2] gy tile free
    uint64_t* done = gempty + 2;            // [1] all MMAs complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.tiles_x * p.tiles_y;
    // accumulator blocks only for the depth taps this launch computes (kd_mask): block index = rank of kd inside the mask
    // ROLES: the CTAs of one launch may split the (gy channel chunk, depth tap) combinations among them (blockIdx % n_roles) and
    // walk the items together -- the x slabs and gy tiles the roles share are then served by L2 instead of one DRAM pass per
    // launch (64 -> 64: six combinations)
    const int role = (int)blockIdx.x % p.n_roles, walker = (int)blockIdx.x / p.n_roles, n_walkers = (int)gridDim.x / p.n_roles;
    const int co0 = p.role_co0[role];
    const unsigned kd_mask = (unsigned)p.role_kd[role];
    const int nkd = __popc(kd_mask & 7u);
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < nkd * KWB * UN) tmem_cols <<= 1;
    auto kd_slot = [&](int kd) { return __popc(kd_mask & ((1u << kd) - 1u)); };

    // zero what TMA never writes: the slab tails (read by the last K step) and the whole gy stages (padding, halo columns)
    {
        const int box_rows = (p.L + 2) * p.BW;
        for (int s = 0; s < kSlots3; ++s) {
            uint4* tail = reinterpret_cast<uint4*>(slab_smem + (size_t)s * p.slab_bytes + (size_t)box_rows * ROWX);
            const int n = (p.slab_bytes - box_rows * ROWX) / 16;
            for (int i = threadIdx.x; i < n; i += kTcThreads) tail[i] = make_uint4(0, 0, 0, 0);
        }
        uint4* g = reinterpret_cast<uint4*>(gy_smem);
        for (int i = threadIdx.x; i < 2 * p.gy_bytes / 16; i += kTcThreads) g[i] = make_uint4(0, 0, 0, 0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_g) : "memory");
        for (int i = 0; i < kSlots3; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(gfull + i, 1); mbar_init(gempty + i, 1); }
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

    auto decode = [&](int item, int& b, int& d_begin, int& nd, int& x0, int& y0) {
        const int t = item % tiles, r = item / tiles;
        const int c = r % p.nchunks;
        b = r / p.nchunks;
        d_begin = c * p.dchunk;
        nd = min(p.dchunk, p.Do - d_begin);
        x0 = (t % p.tiles_x) * (p.BW - 2);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer: x slabs and gy tiles ================
        const uint32_t box_bytes = (uint32_t)ROWX * p.BW * (p.L + 2);
        const uint32_t line_bytes = (uint32_t)ROWG * (p.BW - 2);
        int gs = 0, gp = 0;
        for (int item = walker; item < p.n_items; item += n_walkers) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            int s = 0;
            for (int d = 0; d < nd; ++d, ++gp) {
                for (; s < nd + 2 && s <= d + 2; ++s, ++gs) {      // input planes needed by gy plane d: s <= d + 2
                    const int slot = gs % kSlots3;
                    if (gs >= kSlots3) mbar_wait(empty + slot, ((gs / kSlots3) - 1) & 1);
                    if (elect_one()) {
                        mbar_expect_tx(full + slot, box_bytes);
                        tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, &tm_x, full + slot, 0, x0 + p.off_w, y0 + p.off_h,
                                    d_begin + p.off_d + s, b);
                    }
                    __syncwarp();
                }
                const int st = gp & 1;
                if (gp >= 2) mbar_wait(gempty + st, ((gp >> 1) - 1) & 1);
                if (elect_one()) {
                    mbar_expect_tx(gfull + st, line_bytes * p.L);
                    for (int j = 0; j < p.L; ++j)      // line j -> rows (2+j)*BW .. (2+j)*BW + BW-3 (out of range => zeros)
                        tma_load_5d(gy_smem + (size_t)st * p.gy_bytes + (size_t)(2 + j) * p.BW * ROWG, &tm_g, gfull + st, co0, x0,
                                    y0 + j, d_begin + d, b);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        const uint64_t da0 = umma_desc_mn<ROWX>(0, ROWX);                        // A atoms: one voxel row apart (kw)
        const uint64_t db0 = umma_desc_mn<ROWG>(0, (uint32_t)(p.BW * ROWG));     // B atoms: one line apart (kh = 2 - n)
        const uint32_t a_hi = (uint32_t)(da0 >> 32), b_hi = (uint32_t)(db0 >> 32);
        const uint32_t slab_lo = (uint32_t)da0 | (smem_u32(slab_smem) >> 4);
        const uint32_t gy_lo = (uint32_t)db0 | (smem_u32(gy_smem) >> 4);
        const uint32_t slab16 = (uint32_t)p.slab_bytes >> 4, gy16 = (uint32_t)p.gy_bytes >> 4;
        int gs0 = 0, gp = 0, landed = 0;
        uint32_t first = 1;                              // the CTA's first gy plane initialises the accumulators
        for (int item = walker; item < p.n_items; item += n_walkers) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int st = gp & 1;
                while (landed <= gs0 + d + 2) { mbar_wait(full + landed % kSlots3, (landed / kSlots3) & 1); ++landed; }
                mbar_wait(gfull + st, (gp >> 1) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t g_lo = gy_lo + (uint32_t)st * gy16;
#pragma unroll
                    for (int kd = 0; kd < 3; ++kd) {
                        if (!(kd_mask >> kd & 1u)) continue;
                        const uint32_t s_lo = slab_lo + (uint32_t)((gs0 + d + kd) % kSlots3) * slab16;
#pragma unroll
                        for (int blk = 0; blk < KWB; ++blk) {
                            const uint32_t d_tmem = tmem_base + (uint32_t)((kd_slot(kd) * KWB + blk) * UN);
                            uint32_t a_lo = s_lo + (uint32_t)((blk * 2 * ROWX) >> 4);      // second block: atoms kw = 2, 3(junk)
                            uint32_t b_lo = g_lo;
                            for (int ks = 0; ks < p.ksteps; ++ks) {
                                umma_bf16_lohi(d_tmem, a_lo, a_hi, b_lo, b_hi, IDESC, (first ^ 1u) | (uint32_t)(ks != 0));
                                a_lo += (uint32_t)(16 * ROWX) >> 4;
                                b_lo += (uint32_t)(16 * ROWG) >> 4;
                            }
                        }
                    }
                    umma_commit(empty + (gs0 + d) % kSlots3);
                    if (d == nd - 1) {
                        umma_commit(empty + (gs0 + nd) % kSlots3);
                        umma_commit(empty + (gs0 + nd + 1) % kSlots3);
                    }
                    umma_commit(gempty + st);
                }
                __syncwarp();
                first = 0;
            }
            gs0 += nd + 2;
        }
        if (elect_one()) umma_commit(done);
        __syncwarp();
    } else {
        // ===================================== epilogue: TMEM -> gW ==============================
        mbar_wait(done, 0);
        tc_fence_after();
        const int q = warp & 3;
        const int row = q * 32 + lane;                   // D row = (kw atom, ci)
        constexpr int ATOMS = 128 / CIN;                 // kw atoms per block
        const int kw_in_blk = row / CIN, ci = row % CIN;
        for (int kd = 0; kd < 3; ++kd) {
            if (!(kd_mask >> kd & 1u)) continue;
#pragma unroll
            for (int blk = 0; blk < KWB; ++blk) {
                const int kw = blk * 2 + kw_in_blk;
                const bool real = kw < 3 && kw_in_blk < ATOMS;
#pragma unroll
                for (int c0 = 0; c0 < UN; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld<16>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((kd_slot(kd) * KWB + blk) * UN + c0), v);
                    tmem_ld_wait();
                    if (real) {
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            const int col = c0 + k, n = col / NCO, co = col % NCO;     // atom n <-> kh = 2 - n
                            if (n < 3 && co0 + co < p.cout) {
                                const int slot = p.tap_map[(kd * 3 + (2 - n)) * 3 + kw];
                                if (slot >= 0)
                                    atomicAdd(p.gw + ((size_t)slot * CIN + ci) * p.cout + co0 + co, __uint_as_float(v[k]));
                            }
                        }
                    }
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

struct WgPlan {
    int BW, L, tiles_x, tiles_y, slab_bytes, gy_bytes;
    double score;
};

WgPlan plan_tiles_wgrad(int Ho, int Wo, int rowx, int rowg, size_t smem_budget) {
    WgPlan best{};
    best.score = -1.0;
    for (int L = 1; L <= 64; ++L) {
        for (int BW = 16; BW <= 256; BW += 8) {                // BW*rowg must be a multiple of 128 (TMA destination of a gy line)
            if ((BW * rowg) % 128) continue;
            const int rows_x = (L + 2) * BW + 32;               // + last K step + junk kw atom
            const int rows_g = (L + 5) * BW + 32;               // 2 zero lines before, the tile, the junk atom's reach after
            const int slab = ((rows_x * rowx) + 1023) / 1024 * 1024;
            const int gyb = ((rows_g * rowg) + 1023) / 1024 * 1024;
            if ((size_t)kSlots3 * slab + 2 * (size_t)gyb + 256 > smem_budget) continue;
            const int tiles_x = (Wo + BW - 3) / (BW - 2), tiles_y = (Ho + L - 1) / L;
            const double eff = (double)Wo * Ho / ((double)tiles_x * tiles_y * (L + 2) * BW);   // useful / reduced rows
            if (eff > best.score) best = WgPlan{BW, L, tiles_x, tiles_y, slab, gyb, eff};
        }
    }
    return best;
}

// x_es: element stride of the x sub-lattice per spatial axis (1 = dense, 2 = a parity class of a stride-2 layer); x points at
// the class's first voxel, (Di, Hi, Wi) are the sub-lattice extents and (Dx, Hx, Wx) those of the allocation it lives in.
template <int CIN, int NCO>
int launch_wgrad(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout, int co0,
                 int off_d, int off_h, int off_w, cudaStream_t st, int x_es = 1, int Dx = 0, int Hx = 0, int Wx = 0,
                 unsigned kd_mask = 7u, const int* tap_map = nullptr, int n_roles = 1, const int* role_co0 = nullptr,
                 const int* role_kd = nullptr, int cin_real = CIN) {
    // cin_real < CIN (stride-1 form only): voxel rows of x hold cin_real channels, the TMA box is CIN wide and the channels beyond
    // the tensor's extent arrive as zeros -- rows cin_real.. of every gw tap come out zero
    if (x_es == 1) { Dx = Di; Hx = Hi; Wx = Wi; }
    constexpr int ROWG = NCO * 2;
    constexpr int ROWX_BOX = CIN * 2;
    const int ROWX = cin_real * 2;
    const size_t smem_budget = 227 * 1024 - 1024;
    const WgPlan tp = plan_tiles_wgrad(Ho, Wo, ROWX_BOX, ROWG, smem_budget);
    MVS_REQUIRE(tp.score > 0, "conv3d_s1_wgrad: no slab geometry fits shared memory (Cin=%d, N=%d)", CIN, NCO);

    CUtensorMap tm_x, tm_g;
    {
        const cuuint64_t dims[5] = {(cuuint64_t)cin_real, (cuuint64_t)Wi, (cuuint64_t)Hi, (cuuint64_t)Di, (cuuint64_t)B};
        const cuuint64_t strides[4] = {(cuuint64_t)x_es * ROWX, (cuuint64_t)x_es * ROWX * Wx, (cuuint64_t)x_es * ROWX * Wx * Hx,
                                       (cuuint64_t)ROWX * Wx * Hx * Dx};
        const cuuint32_t box[5] = {(cuuint32_t)CIN, (cuuint32_t)tp.BW, (cuuint32_t)(tp.L + 2), 1, 1};
        MVS_TRY(encode_tiled(&tm_x, x, 5, dims, strides, box, swizzle_for(ROWX_BOX), "conv3d_s1_wgrad", "x"));
    }
    MVS_TRY(encode_volume(&tm_g, gy, cout, NCO, Wo, Ho, Do, B, tp.BW - 2, 1, "conv3d_s1_wgrad", "gy"));
    WgradParams p;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.off_d = off_d; p.off_h = off_h; p.off_w = off_w;
    p.BW = tp.BW; p.L = tp.L; p.tiles_x = tp.tiles_x; p.tiles_y = tp.tiles_y;
    p.cout = cout; p.slab_bytes = tp.slab_bytes; p.gy_bytes = tp.gy_bytes;
    p.n_roles = n_roles;
    for (int r = 0; r < 8; ++r) {
        p.role_co0[r] = role_co0 && r < n_roles ? role_co0[r] : co0;
        p.role_kd[r] = (role_kd && r < n_roles ? role_kd[r] : (int)kd_mask) & 7;
    }
    p.ksteps = ((tp.L + 2) * tp.BW + 15) / 16;
    for (int t = 0; t < 27; ++t) p.tap_map[t] = tap_map ? tap_map[t] : t;
    p.gw = gw;
    const long tiles = (long)tp.tiles_x * tp.tiles_y;
    const int sms = sm_count();
    long walkers = sms / n_roles > 0 ? sms / n_roles : 1;          // CTAs that walk the items (each role has that many)
    {
        // every CTA ends with red.global.add of its whole accumulator set (up to 27 x CIN x NCO floats) onto the same addresses: on a
        // small problem (the 2D networks' maps) a full grid of one-tile CTAs spends its time in those same-address reductions --
        // give every CTA at least kMinPlaneTiles plane tiles of work
        static const long kMinPlaneTiles = [] { const char* e = getenv("MVSB200_WG_MIN_TILES"); return e ? atol(e) : 8L; }();
        const long potential = tiles * B * Do;
        const long cap = potential / (kMinPlaneTiles > 0 ? kMinPlaneTiles : 1);
        if (cap < walkers) walkers = cap > 0 ? cap : 1;
    }
    const Runs runs = choose_runs(tiles, B, Do, walkers, 4);
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    p.n_items = (int)(tiles * p.nchunks * B);
    const dim3 grid((unsigned)((p.n_items < walkers ? p.n_items : walkers) * n_roles), 1, 1);
    const size_t smem = 1024 + (size_t)kSlots3 * tp.slab_bytes + 2 * (size_t)tp.gy_bytes + 256;
    MVS_CUDA(cudaFuncSetAttribute(conv3d_s1_wgrad_tc_kernel<CIN, NCO>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv3d_s1_wgrad_tc_kernel<CIN, NCO><<<grid, kTcThreads, smem, st>>>(tm_x, tm_g, p);
    MVS_CHECK_LAUNCH("conv3d_s1_wgrad_tc");
    return MVSB200_OK;
}

// =================================================================================================================
// Stride-2 convolution forward on tcgen05:  out(o) = sum_k W[k] . x(2o - pad + k)   (per axis, k = 0..2, x zero outside).
// The three stride-2 branches conv_{1,2,3}_0 of the regulariser (scripts/model.py:104-110, stacked along Cout) and, with the
// transposed filter, the data gradient of the transposed convolutions.
// A UMMA operand needs voxel rows at a constant pitch, so the stride-2 reads are turned into stride-1 reads of the four
// in-plane PARITY sub-lattices of x: tap k of an axis reads sub-lattice q = (k - pad) & 1 at index o + s,
// s = (k - pad - q) / 2 in {-1, 0}.  Each sub-lattice is just another 5-D TMA tensor map over the same memory (doubled
// h/w strides, shifted base), so TMA lands parity-pure slabs with a 1-voxel halo; the depth axis needs no
// de-interleaving (plane 2*od - pad + kd is addressed directly).  The slabs form a linear stream -- per output plane:
// 4 parity classes x 3 depth taps -- each consumed once by the 1, 2 or 4 taps that live on it, all accumulating into
// the plane's TMEM accumulator.
constexpr int kS2Slots = 4;

struct ConvS2Params {
    int B, Do, Ho, Wo;              // output volume
    int pad_d, pad_h, pad_w;        // out(o) reads x(2o - pad + k)
    int Dx;                         // input planes (depth is not de-interleaved: out-of-range planes are zero)
    int BW, L, MB;                  // sub-slab: BW voxels per line (incl. 1 halo), L output lines, MB 128-row blocks
    int tiles_x, tiles_y;
    int dchunk, nchunks, n_items;
    int cout, y_cs, y_coff, n_rows, w_row0;
    int slab_bytes;
    __nv_bfloat16* y;
    float* stats;                   // null, or [gridDim.x][2][stats_cs]: per-CTA sums of the outputs and of their squares (fp32
    int stats_cs;                   // accumulators), this launch's channels at column y_coff -- the box BatchNorm that follows the
                                    // stacked branches (scripts/model.py:104-110) then needs no pass over them for its statistics
};

template <int CIN, int NOUT, bool STATS = false>
__global__ void __launch_bounds__(kTcThreads, 1)
conv3d_s2_tc_kernel(const __grid_constant__ CUtensorMap tm_x00, const __grid_constant__ CUtensorMap tm_x01,
                    const __grid_constant__ CUtensorMap tm_x10, const __grid_constant__ CUtensorMap tm_x11,
                    const __grid_constant__ CUtensorMap tm_w, const ConvS2Params p) {
    constexpr int ROWB = CIN * 2;
    constexpr int KSTEPS = CIN / 16;
    constexpr int W_TAP_BYTES = NOUT * ROWB;
    constexpr int W_BYTES = 27 * W_TAP_BYTES;
    constexpr int W_BYTES_AL = (W_BYTES + 1023) / 1024 * 1024;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NOUT >> 3) << 17) | ((128u >> 4) << 24);

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* w_smem = smem;
    unsigned char* slab_smem = smem + W_BYTES_AL;
    uint64_t* bars = reinterpret_cast<uint64_t*>(slab_smem + (size_t)kS2Slots * p.slab_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + kS2Slots;
    uint64_t* wfull = bars + 2 * kS2Slots;
    uint64_t* tfull = wfull + 1;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int MB = p.MB;
    const int tiles = p.tiles_x * p.tiles_y;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * MB * NOUT) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x00) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x01) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x10) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x11) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w) : "memory");
        for (int i = 0; i < kS2Slots; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
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
        nd = min(p.dchunk, p.Do - d_begin);
        x0 = (t % p.tiles_x) * (p.BW - 1);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            mbar_expect_tx(wfull, W_BYTES);
            for (int tap = 0; tap < 27; ++tap)
                tma_load_2d(w_smem + tap * W_TAP_BYTES, &tm_w, wfull, 0, tap * p.n_rows + p.w_row0);
        }
        __syncwarp();
        const uint32_t box_bytes = (uint32_t)ROWB * p.BW * (p.L + 1);
        int gs = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d) {
                for (int c = 0; c < 4; ++c) {
                    const CUtensorMap* tm = c == 0 ? &tm_x00 : (c == 1 ? &tm_x01 : (c == 2 ? &tm_x10 : &tm_x11));
                    for (int kd = 0; kd < 3; ++kd, ++gs) {
                        const int slot = gs % kS2Slots;
                        if (gs >= kS2Slots) mbar_wait(empty + slot, ((gs / kS2Slots) - 1) & 1);
                        if (elect_one()) {
                            mbar_expect_tx(full + slot, box_bytes);
                            tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, tm, full + slot, 0, x0 - 1, y0 - 1,
                                        2 * (d_begin + d) - p.pad_d + kd, b);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        mbar_wait(wfull, 0);
        const uint64_t d0 = umma_desc<ROWB>(0);
        const uint32_t desc_hi = (uint32_t)(d0 >> 32);
        const uint32_t w_lo = (uint32_t)d0 | (smem_u32(w_smem) >> 4);
        const uint32_t slab_lo = (uint32_t)d0 | (smem_u32(slab_smem) >> 4);
        const uint32_t bw16 = (uint32_t)(p.BW * ROWB) >> 4, slab16 = (uint32_t)p.slab_bytes >> 4;
        int gs = 0, gp = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                if (gp >= 2) mbar_wait(tempty + stage, ((gp >> 1) - 1) & 1);
                uint32_t acc = 0;                        // uniform over the 128-row blocks: the plane's first MMA initialises
                for (int c = 0; c < 4; ++c) {
                    const int qy = c >> 1, qx = c & 1;
                    for (int kd = 0; kd < 3; ++kd, ++gs) {
                        const int slot = gs % kS2Slots;
                        mbar_wait(full + slot, (gs / kS2Slots) & 1);
                        tc_fence_after();
                        if (elect_one()) {
                            const uint32_t s_lo = slab_lo + (uint32_t)slot * slab16;
#pragma unroll
                            for (int kh = 0; kh < 3; ++kh) {
                                if (((kh - p.pad_h) & 1) != qy) continue;
                                const int sy = (kh - p.pad_h - qy) >> 1;           // -1 or 0
#pragma unroll
                                for (int kw = 0; kw < 3; ++kw) {
                                    if (((kw - p.pad_w) & 1) != qx) continue;
                                    const int sx = (kw - p.pad_w - qx) >> 1;
                                    const uint32_t row_lo = s_lo + (uint32_t)(sy + 1) * bw16 + (uint32_t)(((sx + 1) * ROWB) >> 4);
                                    const uint32_t wt_lo = w_lo + (uint32_t)((((kd * 3 + kh) * 3 + kw) * W_TAP_BYTES) >> 4);
                                    for (int mb = 0; mb < MB; ++mb) {
                                        const uint32_t d_tmem = tmem_base + (uint32_t)((stage * MB + mb) * NOUT);
#pragma unroll
                                        for (int k = 0; k < KSTEPS; ++k)
                                            umma_bf16_lohi(d_tmem, row_lo + (uint32_t)((mb * 128 * ROWB + k * 32) >> 4), desc_hi,
                                                           wt_lo + (uint32_t)((k * 32) >> 4), desc_hi, IDESC, acc | (uint32_t)(k != 0));
                                    }
                                    acc = 1;
                                }
                            }
                            umma_commit(empty + slot);
                        }
                        __syncwarp();
                        acc = 1;                         // every (class, kd) slab carries at least one tap
                    }
                }
                if (elect_one()) umma_commit(tfull + stage);
                __syncwarp();
            }
        }
    } else {
        // ===================================== epilogue =========================================
        const int q = warp & 3;
        int ti[kMaxMB], tj[kMaxMB];
        bool ok[kMaxMB];
#pragma unroll
        for (int mb = 0; mb < kMaxMB; ++mb) {
            const int m = mb * 128 + q * 32 + lane;
            tj[mb] = m / p.BW; ti[mb] = m - tj[mb] * p.BW;
            ok[mb] = ti[mb] < p.BW - 1 && tj[mb] < p.L;
        }
        constexpr bool want_stats = STATS;            // (a template parameter: 128 more live registers only where they are used)
        float st_s[STATS ? NOUT : 1], st_q[STATS ? NOUT : 1];
#pragma unroll
        for (int ch = 0; ch < (STATS ? NOUT : 1); ++ch) { st_s[ch] = 0.f; st_q[ch] = 0.f; }
        int gp = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                mbar_wait(tfull + stage, (gp >> 1) & 1);
                tc_fence_after();
                __nv_bfloat16* plane0 = p.y + ((((size_t)b * p.Do + d_begin + d) * p.Ho + y0) * p.Wo + x0) * p.y_cs + p.y_coff;
#pragma unroll
                for (int mb = 0; mb < kMaxMB; ++mb) {
                    if (mb < MB) {
#pragma unroll
                        for (int c0 = 0; c0 < NOUT; c0 += 16) {
                            uint32_t v[16];
                            tmem_ld<16>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((stage * MB + mb) * NOUT + c0), v);
                            tmem_ld_wait();
                            if (ok[mb] && x0 + ti[mb] < p.Wo && y0 + tj[mb] < p.Ho) {
                                __nv_bfloat16* row = plane0 + ((size_t)tj[mb] * p.Wo + ti[mb]) * p.y_cs;
                                if constexpr (STATS) {
#pragma unroll
                                    for (int c = 0; c < 16; ++c) {
                                        const float r = __uint_as_float(v[c]);
                                        st_s[c0 + c] += r;
                                        st_q[c0 + c] = fmaf(r, r, st_q[c0 + c]);
                                    }
                                }
#pragma unroll
                                for (int c = 0; c < 16; c += 8) {
                                    if (c0 + c < p.cout) {
                                        const uint4 o = make_uint4(pack_bf16x2(__uint_as_float(v[c]), __uint_as_float(v[c + 1])),
                                                                   pack_bf16x2(__uint_as_float(v[c + 2]), __uint_as_float(v[c + 3])),
                                                                   pack_bf16x2(__uint_as_float(v[c + 4]), __uint_as_float(v[c + 5])),
                                                                   pack_bf16x2(__uint_as_float(v[c + 6]), __uint_as_float(v[c + 7])));
                                        *reinterpret_cast<uint4*>(row + c0 + c) = o;
                                    }
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
        if constexpr (STATS) {
            // warp totals (fixed shuffle order); the four epilogue warps' rows side by side in the slab ring, which is idle by now
            // (the last accumulator has been read: every slab was consumed, every TMA load had landed)
            float* stats_smem = reinterpret_cast<float*>(slab_smem);        // [4 warps][2][NOUT]
#pragma unroll
            for (int ch = 0; ch < NOUT; ++ch) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    st_s[ch] += __shfl_xor_sync(0xffffffffu, st_s[ch], o);
                    st_q[ch] += __shfl_xor_sync(0xffffffffu, st_q[ch], o);
                }
            }
            if (lane == 0) {
#pragma unroll
                for (int ch = 0; ch < NOUT; ++ch) { stats_smem[(q * 2 + 0) * NOUT + ch] = st_s[ch]; stats_smem[(q * 2 + 1) * NOUT + ch] = st_q[ch]; }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (STATS && (int)threadIdx.x < 2 * p.cout) {                       // the CTA's partial row, warps added in fixed order
        const float* stats_smem = reinterpret_cast<const float*>(slab_smem);
        const int which = threadIdx.x / p.cout, ch = threadIdx.x % p.cout;
        float t = 0.f;
#pragma unroll
        for (int w4 = 0; w4 < 4; ++w4) t += stats_smem[(w4 * 2 + which) * NOUT + ch];
        p.stats[((size_t)blockIdx.x * 2 + which) * p.stats_cs + p.y_coff + ch] = t;
    }
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

// partial rows [n_blocks][2][C] of a stride-2 convolution's epilogue statistics -> sums [2][C] (fixed order, fp64 inside)
__global__ void s2_stats_finalize_kernel(const float* __restrict__ partials, int n_blocks, int C, float* __restrict__ sums) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * C) return;
    double acc = 0.0;
    for (int b = 0; b < n_blocks; ++b) acc += (double)partials[(size_t)b * 2 * C + t];
    sums[t] = (float)acc;
}

// stats: null, or the per-CTA statistics rows [grid][2][stats_cs] of the epilogue (ConvS2Params); the launch's grid size is
// then raised into *n_blocks
template <int CIN, int NOUT>
int launch_conv_s2(const void* x, const void* w, void* y, int B, int Dx, int Hx, int Wx, int Do, int Ho, int Wo, int cout, int y_cs,
                   int y_coff, int n_rows, int w_row0, int pad_d, int pad_h, int pad_w, cudaStream_t st, int cin_real, float* stats,
                   int stats_cs, int* n_blocks) {
    // cin_real < CIN: voxel rows of x hold cin_real channels; the TMA box is CIN wide and the channels beyond the tensor's
    // extent arrive as zeros (out-of-bounds fill), so an 8-channel volume feeds the K = 16 MMA without a widened copy
    constexpr int ROWB = CIN * 2;
    const int rowx = cin_real * 2;
    constexpr size_t W_BYTES_AL = ((size_t)27 * NOUT * ROWB + 1023) / 1024 * 1024;
    const size_t smem_budget = 227 * 1024 - 1024;
    const TilePlan tp = plan_tiles(Ho, Wo, ROWB, W_BYTES_AL, smem_budget, kS2Slots, 1, 9, 1);
    MVS_REQUIRE(tp.score > 0, "conv3d_s2: no slab geometry fits shared memory (Cin=%d, N=%d)", CIN, NOUT);

    CUtensorMap tm_x[4], tm_w;
    for (int c = 0; c < 4; ++c) {
        const int qy = c >> 1, qx = c & 1;
        const int Ws = (Wx - qx + 1) / 2, Hs = (Hx - qy + 1) / 2;      // sub-lattice extents
        const char* base = reinterpret_cast<const char*>(x) + ((size_t)qy * Wx + qx) * rowx;
        if (Ws < 1 || Hs < 1) {                                        // degenerate (1-voxel axis): alias class 0, taps read zeros? never used
            tm_x[c] = tm_x[0];
            continue;
        }
        const cuuint64_t dims[5] = {(cuuint64_t)cin_real, (cuuint64_t)Ws, (cuuint64_t)Hs, (cuuint64_t)Dx, (cuuint64_t)B};
        const cuuint64_t strides[4] = {(cuuint64_t)2 * rowx, (cuuint64_t)2 * rowx * Wx, (cuuint64_t)rowx * Wx * Hx,
                                       (cuuint64_t)rowx * Wx * Hx * Dx};
        const cuuint32_t box[5] = {(cuuint32_t)CIN, (cuuint32_t)tp.BW, (cuuint32_t)(tp.L + 1), 1, 1};
        MVS_TRY(encode_tiled(&tm_x[c], base, 5, dims, strides, box, swizzle_for(ROWB), "conv3d_s2", "x, class", c));
    }
    MVS_TRY(encode_filter(&tm_w, w, CIN, 27 * n_rows, NOUT, "conv3d_s2", "w"));
    ConvS2Params p;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.pad_d = pad_d; p.pad_h = pad_h; p.pad_w = pad_w; p.Dx = Dx;
    p.BW = tp.BW; p.L = tp.L; p.MB = tp.MB; p.tiles_x = tp.tiles_x; p.tiles_y = tp.tiles_y;
    p.cout = cout; p.y_cs = y_cs; p.y_coff = y_coff; p.n_rows = n_rows; p.w_row0 = w_row0;
    p.slab_bytes = tp.slab_bytes;
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.stats = stats;
    p.stats_cs = stats_cs;
    MVS_REQUIRE(p.stats == nullptr || (size_t)kS2Slots * tp.slab_bytes >= (size_t)4 * 2 * NOUT * sizeof(float), "conv3d_s2: slab ring too small for the statistics rows");
    MVS_REQUIRE(p.stats == nullptr || 2 * cout <= kTcThreads, "conv3d_s2: %d channels per launch with statistics", cout);
    const long tiles = (long)tp.tiles_x * tp.tiles_y;
    const int sms = sm_count();
    const Runs runs = choose_runs(tiles, B, Do, sms, 1);
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    p.n_items = (int)(tiles * p.nchunks * B);
    const dim3 grid((unsigned)(p.n_items < sms ? p.n_items : sms), 1, 1);
    if (n_blocks && (int)grid.x > *n_blocks) *n_blocks = (int)grid.x;
    const size_t smem = 1024 + W_BYTES_AL + (size_t)kS2Slots * tp.slab_bytes + 256;
    if (p.stats != nullptr) {
        // epilogue statistics: instantiated for the cost volume's 32 channels (the stacked branches, scripts/model.py:104-110)
        if constexpr (CIN == 32) {
            MVS_CUDA(cudaFuncSetAttribute(conv3d_s2_tc_kernel<CIN, NOUT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            conv3d_s2_tc_kernel<CIN, NOUT, true><<<grid, kTcThreads, smem, st>>>(tm_x[0], tm_x[1], tm_x[2], tm_x[3], tm_w, p);
            MVS_CHECK_LAUNCH("conv3d_s2_tc");
            return MVSB200_OK;
        } else {
            MVS_FAIL(MVSB200_E_UNSUPPORTED, "conv3d_s2_fwd_stats: epilogue statistics are built for 32 input channels (got %d)", CIN);
        }
    }
    MVS_CUDA(cudaFuncSetAttribute(conv3d_s2_tc_kernel<CIN, NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv3d_s2_tc_kernel<CIN, NOUT><<<grid, kTcThreads, smem, st>>>(tm_x[0], tm_x[1], tm_x[2], tm_x[3], tm_w, p);
    MVS_CHECK_LAUNCH("conv3d_s2_tc");
    return MVSB200_OK;
}


// =================================================================================================================
// Stride-1 convolution with the DEPTH TAP FOLDED INTO N ("kdn" form).  conv3d_s1_tc_kernel above issues 27 MMAs of N = Cout
// per 128 voxel rows and K step; at N = 16..32 each of them re-reads its 128-row A operand from shared memory for very few
// columns, and the kernel sits on the shared-memory operand-feed roof (profiles/r01_k3_notes.md).  Here the three depth
// taps of a filter become three column blocks of ONE MMA: for an input plane s,
//     Q_s[v, (kd, co)] = sum_{kh,kw,ci} x_s[v + (kh,kw)][ci] * W[kd,kh,kw][ci][co]          (9 MMAs of N = 3 Cout per K step)
// and an output plane is the sum of three such partial planes, out_d = Q_d[kd=0] + Q_{d+1}[kd=1] + Q_{d+2}[kd=2], which the
// epilogue thread that owns the voxel row keeps as two running partial sums in registers while the CTA marches along depth
// (the row of a voxel is the same TMEM lane in every plane: no cross-lane traffic).  A operand reads drop 3x, every slab is
// consumed by exactly one MMA batch (the ring only has to cover the TMA latency), the flops per shared-memory byte of an MMA
// rise 2.1x at Cin = Cout = 32.
struct KdnParams {
    ConvParams c;
    int slots;                      // slab ring depth (2 or 3)
    int planar;                     // 1: the planes are independent maps (2D convolution, mvsb200_conv2d_rows_fwd): only the middle
                                    // depth slice of the filter exists -- MMAs of N = Cout on its row block, one slab per output
                                    // plane (no halo planes), the accumulator IS the output plane (no running partial sums)
    const float* scale;             // AFF: y = relu(acc * scale[c] + shift[c]) per stored channel c of the launch's row block
    const float* shift;             // (fp32 [cout] vectors, offset to the block's first row), then ONE rounding to bf16
};

// AFF (eval-mode BatchNorm + ReLU folded into the epilogue): scale / shift are read from global memory (L1-resident, 2 x cout
// floats) per 8-channel store, after the TMEM load of the slab -- never held across the epilogue, whose volume mode already runs
// near the register limit on its running partial sums.
template <int CIN, int NOUT, int MB, bool AFF = false>
__global__ void __launch_bounds__(kTcThreads, 1)
conv3d_s1_kdn_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                     const __grid_constant__ KdnParams kp) {
    const ConvParams& p = kp.c;
    constexpr int ROWB = CIN * 2;
    constexpr int KSTEPS = CIN / 16;
    constexpr int N3 = 3 * NOUT;
    constexpr int W_TAP_BYTES = NOUT * ROWB;
    constexpr int W_BYTES = 27 * W_TAP_BYTES;
    constexpr int W_BYTES_AL = (W_BYTES + 1023) / 1024 * 1024;
    constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N3 >> 3) << 17) | ((128u >> 4) << 24);
    constexpr uint32_t IDESC_PLANAR = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NOUT >> 3) << 17) | ((128u >> 4) << 24);
    const bool planar = kp.planar != 0;
    const int halo = planar ? 0 : 2;                     // slabs beyond the output planes of a depth run
    constexpr uint32_t TMEM_COLS = 2 * MB * N3 <= 256 ? 256 : 512;
    static_assert(2 * MB * N3 <= 512 && N3 % 16 == 0 && N3 <= 256, "accumulator columns");
    constexpr int kMaxSlots = 3;

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* w_smem = smem;
    unsigned char* slab_smem = smem + W_BYTES_AL;
    const int slots = kp.slots;
    uint64_t* bars = reinterpret_cast<uint64_t*>(slab_smem + (size_t)slots * p.slab_bytes);
    uint64_t* full = bars;                  // [kMaxSlots]
    uint64_t* empty = bars + kMaxSlots;     // [kMaxSlots]
    uint64_t* wfull = bars + 2 * kMaxSlots;
    uint64_t* tfull = wfull + 1;            // [2]
    uint64_t* tempty = tfull + 2;           // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.tiles_x * p.tiles_y;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w) : "memory");
        for (int i = 0; i < kMaxSlots; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
        mbar_init(wfull, 1);
        for (int i = 0; i < 2; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(TMEM_COLS) : "memory");
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
        nd = min(p.dchunk, p.Do - d_begin);
        x0 = (t % p.tiles_x) * (p.BW - 2);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            mbar_expect_tx(wfull, 27u * W_TAP_BYTES);
            // packed as [(kh,kw)][kd][n_rows][Cin]: the three depth taps of an in-plane tap are consecutive row blocks
            for (int t = 0; t < 27; ++t) tma_load_2d(w_smem + t * W_TAP_BYTES, &tm_w, wfull, 0, t * p.n_rows + p.w_row0);
        }
        __syncwarp();
        const uint32_t box_bytes = (uint32_t)ROWB * p.BW * (p.L + 2);
        int gs = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + halo; ++s, ++gs) {
                const int slot = gs % slots;
                if (gs >= slots) mbar_wait(empty + slot, ((gs / slots) - 1) & 1);
                if (elect_one()) {
                    mbar_expect_tx(full + slot, box_bytes);
                    tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, &tm_x, full + slot, 0, x0 + p.off_w, y0 + p.off_h,
                                d_begin + p.off_d + s, b);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        mbar_wait(wfull, 0);
        const uint64_t d0 = umma_desc<ROWB>(0);
        const uint32_t desc_hi = (uint32_t)(d0 >> 32);
        const uint32_t w_lo = (uint32_t)d0 | (smem_u32(w_smem) >> 4);
        const uint32_t slab_lo = (uint32_t)d0 | (smem_u32(slab_smem) >> 4);
        const uint32_t bw16 = (uint32_t)(p.BW * ROWB) >> 4, slab16 = (uint32_t)p.slab_bytes >> 4;
        const uint32_t idesc = planar ? IDESC_PLANAR : IDESC;
        const uint32_t w_kd = planar ? (uint32_t)W_TAP_BYTES >> 4 : 0u;      // planar: the kd = 1 row block of every in-plane tap
        int gs = 0;                                      // slabs processed (all items): ring slot, TMEM stage and phases
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + halo; ++s, ++gs) {
                const int stage = gs & 1, slot = gs % slots;
                if (gs >= 2) mbar_wait(tempty + stage, ((gs >> 1) - 1) & 1);
                mbar_wait(full + slot, (gs / slots) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t slot_lo = slab_lo + (uint32_t)slot * slab16;
#pragma unroll
                    for (int mb = 0; mb < MB; ++mb) {
                        const uint32_t d_tmem = tmem_base + (uint32_t)((stage * MB + mb) * N3);
                        const uint32_t mb16 = (uint32_t)(mb * 128 * ROWB) >> 4;
                        uint32_t acc = 0;
#pragma unroll
                        for (int kh = 0; kh < 3; ++kh) {
                            const uint32_t row_lo = slot_lo + mb16 + kh * bw16;
#pragma unroll
                            for (int kw = 0; kw < 3; ++kw) {
#pragma unroll
                                for (int k = 0; k < KSTEPS; ++k) {
                                    umma_bf16_lohi(d_tmem, row_lo + (uint32_t)((kw * ROWB + k * 32) >> 4), desc_hi,
                                                   w_lo + w_kd + (uint32_t)(((kh * 3 + kw) * 3 * W_TAP_BYTES + k * 32) >> 4), desc_hi, idesc, acc);
                                    acc = 1;
                                }
                            }
                        }
                    }
                    umma_commit(empty + slot);           // this slab is read by this batch only
                    umma_commit(tfull + stage);
                }
                __syncwarp();
            }
        }
    } else {
        // ===================================== epilogue =========================================
        const int q = warp & 3;
        int ti[MB], tj[MB];
        bool in_tile[MB];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
            const int m = mb * 128 + q * 32 + lane;
            tj[mb] = m / p.BW; ti[mb] = m - tj[mb] * p.BW;
            in_tile[mb] = ti[mb] < p.BW - 2 && tj[mb] < p.L;
        }
        float P1[MB][NOUT], P2[MB][NOUT];                // partial sums of output planes s and s-1 (this thread's voxel rows)
        int gs = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + halo; ++s, ++gs) {
                const int stage = gs & 1;
                mbar_wait(tfull + stage, (gs >> 1) & 1);
                tc_fence_after();
                const bool store = s >= halo;            // output plane s - 2 is complete with this slab's kd = 2 block (planar: plane s)
                __nv_bfloat16* plane0 = p.y + (long long)b * p.y_sb + (long long)(d_begin + s - halo) * p.y_sd + (long long)y0 * p.y_sh +
                                        (long long)x0 * p.y_sw + p.y_coff;
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) {
                    const uint32_t t0 = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((stage * MB + mb) * N3);
                    const bool ok = store && in_tile[mb] && x0 + ti[mb] < p.Wo && y0 + tj[mb] < p.Ho;
                    __nv_bfloat16* row = plane0 + (long long)tj[mb] * p.y_sh + (long long)ti[mb] * p.y_sw;
#pragma unroll
                    for (int c0 = 0; c0 < NOUT; c0 += 16) {
                        float o[16];
                        if (planar) {
                            uint32_t v[16];
                            tmem_ld<16>(t0 + (uint32_t)c0, v);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 16; ++i) o[i] = __uint_as_float(v[i]);
                        } else {
                            uint32_t v2[16], v1[16], v0[16];
                            tmem_ld<16>(t0 + (uint32_t)(2 * NOUT + c0), v2);
                            tmem_ld<16>(t0 + (uint32_t)(NOUT + c0), v1);
                            tmem_ld<16>(t0 + (uint32_t)c0, v0);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                o[i] = P2[mb][c0 + i] + __uint_as_float(v2[i]);
                                P2[mb][c0 + i] = P1[mb][c0 + i] + __uint_as_float(v1[i]);
                                P1[mb][c0 + i] = __uint_as_float(v0[i]);
                            }
                        }
                        if (ok) {
#pragma unroll
                            for (int i = 0; i < 16; i += 8) {
                                if (c0 + i < p.cout) {
                                    if constexpr (AFF) {
#pragma unroll
                                        for (int j = 0; j < 8; ++j)
                                            o[i + j] = fmaxf(fmaf(o[i + j], kp.scale[c0 + i + j], kp.shift[c0 + i + j]), 0.f);
                                    }
                                    const uint4 u = make_uint4(pack_bf16x2(o[i], o[i + 1]), pack_bf16x2(o[i + 2], o[i + 3]),
                                                               pack_bf16x2(o[i + 4], o[i + 5]), pack_bf16x2(o[i + 6], o[i + 7]));
                                    *reinterpret_cast<uint4*>(row + c0 + i) = u;
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
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// planar: KdnParams::planar
template <int CIN, int NOUT, int MB, bool AFF>
int launch_conv_kdn_mb(const void* x, const void* w, void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout,
                       int y_cs, int y_coff, int n_rows, int w_row0, int off_d, int off_h, int off_w, const TilePlan& tp, int slots,
                       int planar, cudaStream_t st, int cin_real, const float* scale, const float* shift) {
    // cin_real < CIN: voxel rows of x hold cin_real channels; the TMA box is CIN wide, the channels beyond the tensor's extent
    // arrive as zeros (out-of-bounds fill) -- an 8-channel volume feeds the K = 16 MMA without a widened copy
    constexpr int ROWB = CIN * 2;
    constexpr size_t W_BYTES_AL = ((size_t)27 * NOUT * ROWB + 1023) / 1024 * 1024;
    CUtensorMap tm_x, tm_w;
    MVS_TRY(encode_volume(&tm_x, x, cin_real, CIN, Wi, Hi, Di, B, tp.BW, tp.L + 2, "conv3d_s1_kdn", "x"));
    MVS_TRY(encode_filter(&tm_w, w, CIN, 27 * n_rows, NOUT, "conv3d_s1_kdn", "w"));
    KdnParams kp;
    ConvParams& p = kp.c;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo;
    p.off_d = off_d; p.off_h = off_h; p.off_w = off_w;
    p.BW = tp.BW; p.L = tp.L; p.MB = MB; p.tiles_x = tp.tiles_x; p.tiles_y = tp.tiles_y;
    p.cout = cout; p.y_cs = y_cs; p.y_coff = y_coff; p.n_rows = n_rows; p.w_row0 = w_row0;
    p.slab_bytes = tp.slab_bytes;
    p.tap_mask = 0x7ffffffu;
    p.y_sw = y_cs; p.y_sh = (long long)Wo * y_cs; p.y_sd = (long long)Ho * Wo * y_cs; p.y_sb = (long long)Do * Ho * Wo * y_cs;
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    kp.slots = slots;
    kp.planar = planar;
    kp.scale = AFF ? scale + y_coff : nullptr;
    kp.shift = AFF ? shift + y_coff : nullptr;
    const int halo = planar ? 0 : 2;
    const long tiles = (long)tp.tiles_x * tp.tiles_y;
    const int sms = sm_count();
    const Runs runs = choose_runs(tiles, B, Do, sms, halo + 1);      // nd + 2 slabs per run (planar: nd) + pipeline fill
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    p.n_items = (int)(tiles * p.nchunks * B);
    const dim3 grid((unsigned)(p.n_items < sms ? p.n_items : sms), 1, 1);
    const size_t smem = 1024 + W_BYTES_AL + (size_t)slots * tp.slab_bytes + 256;
    MVS_CUDA(cudaFuncSetAttribute(conv3d_s1_kdn_kernel<CIN, NOUT, MB, AFF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    conv3d_s1_kdn_kernel<CIN, NOUT, MB, AFF><<<grid, kTcThreads, smem, st>>>(tm_x, tm_w, kp);
    MVS_CHECK_LAUNCH("conv3d_s1_kdn");
    return MVSB200_OK;
}

template <int CIN, int NOUT, bool AFF>
int launch_conv_kdn(const void* x, const void* w, void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout,
                    int y_cs, int y_coff, int n_rows, int w_row0, int off_d, int off_h, int off_w, int planar, cudaStream_t st,
                    int cin_real, const float* scale, const float* shift) {
    constexpr int ROWB = CIN * 2;
    constexpr size_t W_BYTES_AL = ((size_t)27 * NOUT * ROWB + 1023) / 1024 * 1024;
    constexpr int MBMAX = 512 / (2 * 3 * NOUT) >= 4 ? 4 : (512 / (2 * 3 * NOUT) >= 2 ? 2 : 1);
    const size_t smem_budget = 227 * 1024 - 1024;
    // slab geometry: the largest block count that fits, with a 3-deep ring if shared memory allows, else 2-deep
    TilePlan best{};
    best.score = -1.0;
    int best_slots = 0;
    for (int MB = MBMAX; MB >= 1; MB /= 2) {
        for (int slots = 3; slots >= 2; --slots) {
            const TilePlan tp = plan_slab(Ho, Wo, ROWB, W_BYTES_AL, smem_budget, MB, slots, 2, 6, 2);
            if (tp.score > best.score * 1.02 || (best_slots == 0 && tp.score > 0)) { best = tp; best_slots = slots; }
            if (tp.score > 0) break;                      // a 3-deep ring fits for this MB: do not consider 2
        }
    }
    MVS_REQUIRE(best.score > 0, "conv3d_s1_kdn: no slab geometry fits shared memory (Cin=%d, N=%d)", CIN, NOUT);
    auto run = [&](auto mb) {
        return launch_conv_kdn_mb<CIN, NOUT, decltype(mb)::value, AFF>(x, w, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, y_cs, y_coff, n_rows,
                                                                      w_row0, off_d, off_h, off_w, best, best_slots, planar, st,
                                                                      cin_real, scale, shift);
    };
    if (best.MB == 1) return run(std::integral_constant<int, 1>{});
    if constexpr (MBMAX >= 2) { if (best.MB == 2) return run(std::integral_constant<int, 2>{}); }
    if constexpr (MBMAX >= 4) { if (best.MB == 4) return run(std::integral_constant<int, 4>{}); }
    MVS_FAIL(MVSB200_E_UNSUPPORTED, "conv3d_s1_kdn: block count %d", best.MB);
}

// =================================================================================================================
// Stride-2 TRANSPOSED convolution (ConvTranspose3d k=3, scripts/model.py:229-234, used at :115-121) in ONE launch.
//   out[2J + par] = sum over the filter taps k with (par + pad - k) even of W[k] . in[J + (par + pad - k)/2]   (per axis)
// i.e. each of the 8 output-parity classes is a stride-1 convolution of the INPUT lattice with a sub-set of the taps, and
// the 8 sub-sets together are exactly the 27 taps.  The forward kernel above, launched once per class, writes every class
// as a stride-2 sub-lattice of the canvas (64-byte pieces 128 bytes apart, each line visited by 8 launches).  Here a CTA
// marches along the input depth once, keeps EIGHT accumulator blocks (one per class) per stage in TMEM, and the epilogue
// interleaves the classes so that a thread writes the two w-parities of a voxel pair back to back: full, contiguous lines
// of the canvas, each written once.  MMAs: ONE PER INPUT SHIFT (8 per K step; DeconvWide in tc_common.cuh) over the range
// of class blocks that read the shift, with zero filter slots for the classes in the range that do not -- the earlier
// form issued one MMA per run of adjacent user classes (14 per K step) and sat on the shared-memory A-operand feed.
constexpr int kDeconvSlots = 31;     // filter slots of the one-MMA-per-shift table (27 taps + zero slots), pads in {1,2}

struct DeconvParams {
    int B, Do, Ho, Wo;              // extent of the canvas that is written (voxels beyond it are dropped)
    int Jd, Jh, Jw;                 // output lattice (voxel octets): ceil(extent / 2)
    int BW, L, MB;
    int tiles_x, tiles_y;
    int dchunk, nchunks, n_items;
    int cout, n_rows;
    int slab_bytes;
    DeconvWide g;                   // one MMA per input shift: Gray-ordered classes, zero filter slots (tc_common.cuh)
    int wide_io;                    // 1: 32-byte stores (rows 32-byte aligned, channels in multiples of 16)
    long long y_sb, y_sd, y_sh, y_sw;   // canvas voxel-row strides in elements
    __nv_bfloat16* y;
    float* stats;                   // null, or [gridDim.x][2][cout]: per-CTA sums of the stored values and of their squares (the
                                    // train-mode BatchNorm that follows takes its statistics from here: no pass over the canvas)
    // EPI only (see deconv3d_s2_tc_kernel): the output window and the eval-mode BatchNorm + ReLU + skip-add epilogue
    int lo_d, lo_h, lo_w;           // canvas voxel at the window's origin; Do / Ho / Wo above are then the window's END
    int j0_d, j0_h, j0_w;           // first voxel octet that meets the window: lo / 2 (Jd / Jh / Jw count the octets from there)
    const float* scale;             // fp32 [cout]
    const float* shift;             // fp32 [cout]
    const __nv_bfloat16* add;       // null, or bf16 rows in the window's frame with y's strides
};

// EPI: eval-mode form.  y = relu(acc * scale[c] + shift[c]) (+ add[voxel][c]), rounded once to bf16, written only on an
// axis-aligned WINDOW [lo, Do) x [lo_h, Ho) x [lo_w, Wo) of the canvas, in the window's frame (voxel lo -> row 0 of y / add).
// Geometry: the kernel's work unit is the voxel octet J (outputs 2J + par, par in {0,1}^3).  The octets issued are those that
// meet the window, J = j0 + j with j0 = floor(lo / 2) and j < Jd = floor((Do - 1) / 2) - j0 + 1 per axis; the input slabs are
// fetched j0 further along.  An odd lo means the first octet's parity-0 voxels lie before the window: like the voxels past
// Do they are computed and not stored.  The MMA schedule (one MMA per input shift) and the 32-byte stores are those of the
// dense form, so the window of a full-canvas launch and a windowed launch store bit-identical values.
template <int CIN, int NOUT, bool EPI = false>
__global__ void __launch_bounds__(kTcThreads, 1)
deconv3d_s2_tc_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w,
                      const __grid_constant__ DeconvParams p) {
    constexpr int ROWB = CIN * 2;
    constexpr int KSTEPS = CIN / 16;
    constexpr int W_TAP_BYTES = NOUT * ROWB;
    constexpr int W_BYTES = kDeconvSlots * W_TAP_BYTES;
    constexpr int W_BYTES_AL = (W_BYTES + 1023) / 1024 * 1024;
    constexpr int MB = 512 / (16 * NOUT);               // 2 stages x MB x 8 classes x NOUT columns == 512
    // instruction descriptor without the N field: D fp32, A/B bf16, both K-major, M = 128; N = ncls * NOUT per group
    constexpr uint32_t IDESC0 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
    static_assert(MB >= 1 && MB <= 2, "accumulator blocks per class");

    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
    unsigned char* w_smem = smem;
    unsigned char* slab_smem = smem + W_BYTES_AL;
    uint64_t* bars = reinterpret_cast<uint64_t*>(slab_smem + (size_t)kSlots3 * p.slab_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + kSlots3;
    uint64_t* wfull = bars + 2 * kSlots3;
    uint64_t* tfull = wfull + 1;
    uint64_t* tempty = tfull + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
    float* stats_smem = reinterpret_cast<float*>(bars + 16);        // [4 warps][2][NOUT]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles = p.tiles_x * p.tiles_y;
    constexpr uint32_t tmem_cols = 512;

    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_w) : "memory");
        for (int i = 0; i < kSlots3; ++i) { mbar_init(full + i, 1); mbar_init(empty + i, 1); }
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
        x0 = (t % p.tiles_x) * (p.BW - 2);
        y0 = (t / p.tiles_x) * p.L;
    };

    if (warp == 0) {
        // ===================================== TMA producer =====================================
        if (elect_one()) {
            mbar_expect_tx(wfull, (uint32_t)p.g.n_slots * W_TAP_BYTES);
            for (int e = 0; e < p.g.n_slots; ++e)      // tap 27 of the packed weights is all zeros
                tma_load_2d(w_smem + e * W_TAP_BYTES, &tm_w, wfull, 0, p.g.tap_k[e] * p.n_rows);
        }
        __syncwarp();
        const uint32_t box_bytes = (uint32_t)ROWB * p.BW * (p.L + 2);
        int gs = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int s = 0; s < nd + 2; ++s, ++gs) {     // input planes d_begin - 1 + s
                const int slot = gs % kSlots3;
                if (gs >= kSlots3) mbar_wait(empty + slot, ((gs / kSlots3) - 1) & 1);
                if (elect_one()) {
                    mbar_expect_tx(full + slot, box_bytes);
                    if constexpr (EPI)
                        tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, &tm_x, full + slot, 0, p.j0_w + x0 - 1, p.j0_h + y0 - 1,
                                    p.j0_d + d_begin - 1 + s, b);
                    else
                        tma_load_5d(slab_smem + (size_t)slot * p.slab_bytes, &tm_x, full + slot, 0, x0 - 1, y0 - 1, d_begin - 1 + s, b);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================================== MMA issuer =======================================
        mbar_wait(wfull, 0);
        const uint64_t d0 = umma_desc<ROWB>(0);
        const uint32_t desc_hi = (uint32_t)(d0 >> 32);
        const uint32_t w_lo = (uint32_t)d0 | (smem_u32(w_smem) >> 4);
        const uint32_t slab_lo = (uint32_t)d0 | (smem_u32(slab_smem) >> 4);
        const uint32_t bw16 = (uint32_t)(p.BW * ROWB) >> 4, slab16 = (uint32_t)p.slab_bytes >> 4;
        int gs0 = 0, gp = 0, landed = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                if (gp >= 2) mbar_wait(tempty + stage, ((gp >> 1) - 1) & 1);
                while (landed <= gs0 + d + 2) { mbar_wait(full + landed % kSlots3, (landed / kSlots3) & 1); ++landed; }
                tc_fence_after();
                if (elect_one()) {
                    uint32_t slot_lo[3];
#pragma unroll
                    for (int kd = 0; kd < 3; ++kd) slot_lo[kd] = slab_lo + (uint32_t)((gs0 + d + kd) % kSlots3) * slab16;
#pragma unroll
                    for (int mb = 0; mb < MB; ++mb) {
                        const uint32_t mb16 = (uint32_t)(mb * 128 * ROWB) >> 4;
                        for (int g = 0; g < p.g.n_groups; ++g) {
                            const int td = p.g.grp_td[g];
                            const uint32_t a_lo = (td == 0 ? slot_lo[0] : (td == 1 ? slot_lo[1] : slot_lo[2])) + mb16 +
                                                  (uint32_t)p.g.grp_th[g] * bw16 + (uint32_t)((p.g.grp_tw[g] * ROWB) >> 4);
                            const uint32_t b_lo = w_lo + (uint32_t)((p.g.grp_slot0[g] * W_TAP_BYTES) >> 4);
                            const uint32_t d_tmem = tmem_base + (uint32_t)(((stage * MB + mb) * 8 + p.g.grp_pos0[g]) * NOUT);
                            const uint32_t idesc = IDESC0 | ((uint32_t)((p.g.grp_npos[g] * NOUT) >> 3) << 17);
                            uint32_t acc = p.g.grp_first[g] ? 0u : 1u;
#pragma unroll
                            for (int k = 0; k < KSTEPS; ++k) {
                                umma_bf16_lohi(d_tmem, a_lo + (uint32_t)((k * 32) >> 4), desc_hi, b_lo + (uint32_t)((k * 32) >> 4), desc_hi,
                                               idesc, acc);
                                acc = 1;
                            }
                        }
                    }
                    umma_commit(empty + (gs0 + d) % kSlots3);
                    if (d == nd - 1) {
                        umma_commit(empty + (gs0 + nd) % kSlots3);
                        umma_commit(empty + (gs0 + nd + 1) % kSlots3);
                    }
                    umma_commit(tfull + stage);
                }
                __syncwarp();
            }
            gs0 += nd + 2;
        }
    } else {
        // ===================================== epilogue =========================================
        const int q = warp & 3;
        int ti[MB], tj[MB];
        bool in_tile[MB];
#pragma unroll
        for (int mb = 0; mb < MB; ++mb) {
            const int m = mb * 128 + q * 32 + lane;
            tj[mb] = m / p.BW; ti[mb] = m - tj[mb] * p.BW;
            in_tile[mb] = ti[mb] < p.BW - 2 && tj[mb] < p.L;
        }
        // EPI: the BatchNorm vectors in registers for the whole epilogue (at most 2 x 32 floats; this kernel has the room, and
        // per-voxel loads of them cost more epilogue issue slots than the stores)
        float e_sc[EPI ? NOUT : 1], e_sh[EPI ? NOUT : 1];
        if constexpr (EPI) {
#pragma unroll
            for (int ch = 0; ch < NOUT; ++ch) {
                e_sc[ch] = ch < p.cout ? p.scale[ch] : 0.f;
                e_sh[ch] = ch < p.cout ? p.shift[ch] : 0.f;
            }
        }
        // per-channel sums of what this thread stores, for the BatchNorm that follows
        float st_s[NOUT], st_q[NOUT];
#pragma unroll
        for (int ch = 0; ch < NOUT; ++ch) { st_s[ch] = 0.f; st_q[ch] = 0.f; }
        const bool want_stats = !EPI && p.stats != nullptr;
        int gp = 0;
        for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
            int b, d_begin, nd, x0, y0;
            decode(item, b, d_begin, nd, x0, y0);
            for (int d = 0; d < nd; ++d, ++gp) {
                const int stage = gp & 1;
                mbar_wait(tfull + stage, (gp >> 1) & 1);
                tc_fence_after();
#pragma unroll
                for (int mb = 0; mb < MB; ++mb) {
                    const int ox = 2 * (x0 + ti[mb]), oy = 2 * (y0 + tj[mb]), oz = 2 * (d_begin + d);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        uint32_t v[NOUT];
                        tmem_ld<NOUT>(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(((stage * MB + mb) * 8 + c) * NOUT), v);
                        tmem_ld_wait();
                        const int cl = p.g.cls_of_pos[c];                  // accumulator block c holds output-parity class cl
                        if constexpr (EPI) {
                            const int z = 2 * p.j0_d + oz + (cl >> 2), yy = 2 * p.j0_h + oy + (cl >> 1 & 1), xx = 2 * p.j0_w + ox + (cl & 1);
                            if (in_tile[mb] && z >= p.lo_d && yy >= p.lo_h && xx >= p.lo_w && z < p.Do && yy < p.Ho && xx < p.Wo) {
                                const long long off = (long long)b * p.y_sb + (long long)(z - p.lo_d) * p.y_sd +
                                                      (long long)(yy - p.lo_h) * p.y_sh + (long long)(xx - p.lo_w) * p.y_sw;
                                // 8 channels ch .. ch + 7: affine, ReLU, skip addition in fp32, one rounding
                                auto epi8 = [&](int ch) {
                                    float a[8];
#pragma unroll
                                    for (int i = 0; i < 8; ++i) a[i] = fmaxf(fmaf(__uint_as_float(v[ch + i]), e_sc[ch + i], e_sh[ch + i]), 0.f);
                                    if (p.add != nullptr) {
                                        const uint4 r = *reinterpret_cast<const uint4*>(p.add + off + ch);
                                        const uint32_t rw[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
                                        for (int i = 0; i < 4; ++i) {
                                            a[2 * i] += __uint_as_float(rw[i] << 16);
                                            a[2 * i + 1] += __uint_as_float(rw[i] & 0xffff0000u);
                                        }
                                    }
                                    return make_uint4(pack_bf16x2(a[0], a[1]), pack_bf16x2(a[2], a[3]), pack_bf16x2(a[4], a[5]),
                                                      pack_bf16x2(a[6], a[7]));
                                };
                                __nv_bfloat16* row = p.y + off;
                                if (p.wide_io) {
#pragma unroll
                                    for (int ch = 0; ch < NOUT; ch += 16) {
                                        if (ch < p.cout) {
                                            const uint4 lo = epi8(ch), hi = epi8(ch + 8);
                                            U8 o;
                                            o.v[0] = lo.x; o.v[1] = lo.y; o.v[2] = lo.z; o.v[3] = lo.w;
                                            o.v[4] = hi.x; o.v[5] = hi.y; o.v[6] = hi.z; o.v[7] = hi.w;
                                            st_u8(row + ch, o);
                                        }
                                    }
                                } else {
#pragma unroll
                                    for (int ch = 0; ch < NOUT; ch += 8)
                                        if (ch < p.cout) *reinterpret_cast<uint4*>(row + ch) = epi8(ch);
                                }
                            }
                            continue;
                        }
                        const int z = oz + (cl >> 2), yy = oy + (cl >> 1 & 1), xx = ox + (cl & 1);
                        if (in_tile[mb] && z < p.Do && yy < p.Ho && xx < p.Wo) {
                            if (want_stats) {
#pragma unroll
                                for (int ch = 0; ch < NOUT; ++ch) {
                                    // (the fp32 accumulator, not its bf16 rounding: the rounding error is unbiased and 2^-9 relative,
                                    // far inside the statistics' own noise; re-rounding here cost more than the pass it saves)
                                    const float r = __uint_as_float(v[ch]);
                                    st_s[ch] += r;
                                    st_q[ch] = fmaf(r, r, st_q[ch]);
                                }
                            }
                            __nv_bfloat16* row = p.y + (long long)b * p.y_sb + (long long)z * p.y_sd + (long long)yy * p.y_sh + (long long)xx * p.y_sw;
                            if (p.wide_io) {                                   // 32-byte stores: half as many store instructions
#pragma unroll
                                for (int ch = 0; ch < NOUT; ch += 16) {
                                    if (ch < p.cout) {
                                        U8 o;
#pragma unroll
                                        for (int i = 0; i < 8; ++i)
                                            o.v[i] = pack_bf16x2(__uint_as_float(v[ch + 2 * i]), __uint_as_float(v[ch + 2 * i + 1]));
                                        st_u8(row + ch, o);
                                    }
                                }
                                continue;
                            }
#pragma unroll
                            for (int ch = 0; ch < NOUT; ch += 8) {
                                if (ch < p.cout) {
                                    const uint4 o = make_uint4(pack_bf16x2(__uint_as_float(v[ch]), __uint_as_float(v[ch + 1])),
                                                               pack_bf16x2(__uint_as_float(v[ch + 2]), __uint_as_float(v[ch + 3])),
                                                               pack_bf16x2(__uint_as_float(v[ch + 4]), __uint_as_float(v[ch + 5])),
                                                               pack_bf16x2(__uint_as_float(v[ch + 6]), __uint_as_float(v[ch + 7])));
                                    *reinterpret_cast<uint4*>(row + ch) = o;
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
        if (want_stats) {
            // warp totals (fixed shuffle order), then the four epilogue warps' rows side by side in shared memory
#pragma unroll
            for (int ch = 0; ch < NOUT; ++ch) {
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    st_s[ch] += __shfl_xor_sync(0xffffffffu, st_s[ch], o);
                    st_q[ch] += __shfl_xor_sync(0xffffffffu, st_q[ch], o);
                }
            }
            if (lane == 0) {
#pragma unroll
                for (int ch = 0; ch < NOUT; ++ch) { stats_smem[(q * 2 + 0) * NOUT + ch] = st_s[ch]; stats_smem[(q * 2 + 1) * NOUT + ch] = st_q[ch]; }
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (p.stats != nullptr && (int)threadIdx.x < 2 * p.cout) {          // the CTA's partial row [2][cout], warps added in fixed order
        const int which = threadIdx.x / p.cout, ch = threadIdx.x % p.cout;
        float t = 0.f;
#pragma unroll
        for (int w4 = 0; w4 < 4; ++w4) t += stats_smem[(w4 * 2 + which) * NOUT + ch];
        p.stats[((size_t)blockIdx.x * 2 + which) * p.cout + ch] = t;
    }
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

// EPI: win (host int[6]: lo_d, lo_h, lo_w, n_d, n_h, n_w) is the window of the Do x Ho x Wo canvas that is written, y / add
// point at its origin; scale / shift / add as in DeconvParams.
template <int CIN, int NOUT, bool EPI = false>
int launch_deconv_s2(const void* x, const void* w, void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout,
                     int n_rows, int pad_d, int pad_h, int pad_w, const long long* y_strides4, cudaStream_t st,
                     float* stats, int* n_blocks_out, const int* win, const float* scale, const float* shift, const void* add) {
    constexpr int ROWB = CIN * 2;
    constexpr int MB = 512 / (16 * NOUT);
    constexpr size_t W_BYTES_AL = ((size_t)kDeconvSlots * NOUT * ROWB + 1023) / 1024 * 1024;
    const size_t smem_budget = 227 * 1024 - 1024 - 1024;      // - the epilogue's statistics rows
    int Jd = (Do + 1) / 2, Jh = (Ho + 1) / 2, Jw = (Wo + 1) / 2;
    if (EPI) {
        Jd = (win[0] + win[3] - 1) / 2 - win[0] / 2 + 1;
        Jh = (win[1] + win[4] - 1) / 2 - win[1] / 2 + 1;
        Jw = (win[2] + win[5] - 1) / 2 - win[2] / 2 + 1;
    }
    const TilePlan tp = plan_slab(Jh, Jw, ROWB, W_BYTES_AL, smem_budget, MB, kSlots3, 2, 6, 2);
    MVS_REQUIRE(tp.score > 0, "deconv3d_s2: no slab geometry fits shared memory (Cin=%d, N=%d)", CIN, NOUT);

    CUtensorMap tm_x, tm_w;
    MVS_TRY(encode_volume(&tm_x, x, CIN, CIN, Wi, Hi, Di, B, tp.BW, tp.L + 2, "deconv3d_s2", "x"));
    MVS_TRY(encode_filter(&tm_w, w, CIN, 28 * n_rows, NOUT, "deconv3d_s2", "w"));      // 27 taps + the all-zero tap

    DeconvParams p;
    p.B = B; p.Do = Do; p.Ho = Ho; p.Wo = Wo; p.Jd = Jd; p.Jh = Jh; p.Jw = Jw;
    p.lo_d = p.lo_h = p.lo_w = p.j0_d = p.j0_h = p.j0_w = 0;
    p.scale = scale; p.shift = shift; p.add = reinterpret_cast<const __nv_bfloat16*>(add);
    if (EPI) {
        p.lo_d = win[0]; p.lo_h = win[1]; p.lo_w = win[2];
        p.j0_d = win[0] / 2; p.j0_h = win[1] / 2; p.j0_w = win[2] / 2;
        p.Do = win[0] + win[3]; p.Ho = win[1] + win[4]; p.Wo = win[2] + win[5];
    }
    p.BW = tp.BW; p.L = tp.L; p.MB = MB; p.tiles_x = tp.tiles_x; p.tiles_y = tp.tiles_y;
    p.cout = cout; p.n_rows = n_rows; p.slab_bytes = tp.slab_bytes;
    MVS_TRY(build_deconv_wide(pad_d, pad_h, pad_w, NOUT, p.g));
    MVS_REQUIRE(p.g.n_slots <= kDeconvSlots, "deconv3d_s2: %d filter slots", p.g.n_slots);
    p.y_sb = y_strides4[0]; p.y_sd = y_strides4[1]; p.y_sh = y_strides4[2]; p.y_sw = y_strides4[3];
    p.y = reinterpret_cast<__nv_bfloat16*>(y);
    p.wide_io = (cout % 16 == 0 && p.y_sb % 16 == 0 && p.y_sd % 16 == 0 && p.y_sh % 16 == 0 && p.y_sw % 16 == 0 && ((uintptr_t)y & 31u) == 0) ? 1 : 0;

    const long tiles = (long)tp.tiles_x * tp.tiles_y;
    const int sms = sm_count();
    const Runs runs = choose_runs(tiles, B, Jd, sms, 4);
    p.nchunks = runs.nchunks;
    p.dchunk = runs.chunk;
    p.n_items = (int)(tiles * p.nchunks * B);
    const dim3 grid((unsigned)(p.n_items < sms ? p.n_items : sms), 1, 1);
    const size_t smem = 1024 + W_BYTES_AL + (size_t)kSlots3 * tp.slab_bytes + 256 + 1024;
    p.stats = stats;
    if (n_blocks_out) *n_blocks_out = (int)grid.x;
    MVS_CUDA(cudaFuncSetAttribute(deconv3d_s2_tc_kernel<CIN, NOUT, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    deconv3d_s2_tc_kernel<CIN, NOUT, EPI><<<grid, kTcThreads, smem, st>>>(tm_x, tm_w, p);
    MVS_CHECK_LAUNCH("deconv3d_s2_tc");
    return MVSB200_OK;
}

// ---- entry points ---------------------------------------------------------------------------------------------
// Channel dispatch: Ch<CI, N> is one instantiated pair of input channels and filter rows per launch; K is the kernel's
// channel width (8-channel voxel rows run on the 16-channel kernel, whose TMA box reads the missing channels as zeros).
template <int CI, int N>
struct Ch { static constexpr int cin = CI, n = N, k = CI < 16 ? 16 : CI; };
template <class... C>
struct ChList {};
using ConvChannels = ChList<Ch<16, 16>, Ch<16, 32>, Ch<32, 16>, Ch<32, 32>, Ch<64, 16>, Ch<64, 32>>;
using KdnChannels = ChList<Ch<8, 16>, Ch<8, 32>, Ch<16, 16>, Ch<16, 32>, Ch<32, 16>, Ch<32, 32>, Ch<64, 16>, Ch<64, 32>>;
using S2Channels = ChList<Ch<8, 16>, Ch<8, 32>, Ch<16, 16>, Ch<16, 32>, Ch<16, 48>, Ch<16, 64>, Ch<32, 16>, Ch<32, 32>, Ch<32, 48>,
                          Ch<32, 64>, Ch<64, 16>, Ch<64, 32>>;
using WgradChannels = ChList<Ch<16, 8>, Ch<16, 16>, Ch<16, 32>, Ch<32, 8>, Ch<32, 16>, Ch<32, 32>, Ch<64, 8>, Ch<64, 16>, Ch<64, 32>>;

// runs f(C{}) for the listed pair C = (cin, n) and returns true with its result in rc; false if no pair is listed
template <class... C, class F>
bool dispatch(ChList<C...>, int cin, int n, int& rc, F&& f) {
    return ((cin == C::cin && n == C::n && ((rc = f(C{})), true)) || ...);
}

// checks of the stride-1 forward entry points (conv3d_s1_fwd, conv3d_s1_fwd_ex and the kdn forms)
int check_s1_fwd(const char* name, const void* x, const void* w, const void* y, int B, int Di, int Hi, int Wi, int Do, int Ho,
                 int Wo, int cout, int y_cs, int n_rows) {
    MVS_TRY(check_pointers(name, {x, w, y}));
    MVS_REQUIRE(B >= 1 && B <= 65535 && Di >= 1 && Hi >= 1 && Wi >= 1 && Do >= 1 && Ho >= 1 && Wo >= 1, "%s: bad shape", name);
    MVS_REQUIRE(cout >= 8 && cout % 8 == 0 && cout <= n_rows && n_rows % 16 == 0 && n_rows <= 64,
                "%s: cout must be a multiple of 8 and n_rows a multiple of 16 <= 64 (cout=%d n_rows=%d)", name, cout, n_rows);
    MVS_REQUIRE(y_cs >= cout && y_cs % 8 == 0, "%s: output channel stride %d", name, y_cs);
    return MVSB200_OK;
}

}  // namespace

static int conv3d_s1_dispatch(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin, int Do, int Ho,
                              int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w, unsigned tap_mask,
                              const long long* y_strides4, cudaStream_t st, const char* name) {
    MVS_TRY(check_s1_fwd(name, x, w_packed, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, y_cs, n_rows));
    MVS_REQUIRE((tap_mask & 0x7ffffffu) != 0, "%s: empty tap mask", name);
    // N (filter rows per launch) is 16 or 32; a 64-row filter runs as two 32-row halves (all 27 taps of a 64 x 64
    // filter do not fit next to the slab ring; at N = 32 the tensor pipe is fed from shared memory at the same rate)
    for (int row0 = 0; row0 < n_rows && row0 < cout; row0 += 32) {
        const int nout = n_rows - row0 < 32 ? n_rows - row0 : 32;
        const int c_here = cout - row0 < nout ? cout - row0 : nout;
        int rc = MVSB200_OK;
        if (!dispatch(ConvChannels{}, Cin, nout, rc, [&](auto c) {
                using C = decltype(c);
                return launch_conv<C::k, C::n>(x, w_packed, y, B, Di, Hi, Wi, Do, Ho, Wo, c_here, y_cs, row0, n_rows, row0, off_d, off_h,
                                               off_w, tap_mask, y_strides4, st);
            }))
            MVS_FAIL(MVSB200_E_UNSUPPORTED, "%s: unsupported channels Cin=%d n_rows=%d", name, Cin, n_rows);
        MVS_TRY(rc);
    }
    return MVSB200_OK;
}

extern "C" int mvsb200_conv3d_s1_fwd(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                     int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                                     void* stream) {
    return conv3d_s1_dispatch(x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, y_cs, n_rows, off_d, off_h, off_w, 0x7ffffffu,
                              nullptr, (cudaStream_t)stream, "conv3d_s1_fwd");
}

extern "C" int mvsb200_conv3d_s1_fwd_ex(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                        int Do, int Ho, int Wo, int cout, int n_rows, int off_d, int off_h, int off_w,
                                        unsigned tap_mask, const int64_t* y_strides4, void* stream) {
    MVS_REQUIRE(y_strides4 != nullptr, "conv3d_s1_fwd_ex: null output strides");
    long long ys[4];
    MVS_TRY(copy_strides("conv3d_s1_fwd_ex", y_strides4, ys));
    return conv3d_s1_dispatch(x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, cout, n_rows, off_d, off_h, off_w, tap_mask, ys,
                              (cudaStream_t)stream, "conv3d_s1_fwd_ex");
}

extern "C" int mvsb200_conv3d_s1_wgrad_ex(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Cin, int Do,
                                          int Ho, int Wo, int cout, int off_d, int off_h, int off_w, unsigned kd_mask, void* stream);

extern "C" int mvsb200_conv3d_s1_wgrad(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Cin, int Do,
                                       int Ho, int Wo, int cout, int off_d, int off_h, int off_w, void* stream) {
    return mvsb200_conv3d_s1_wgrad_ex(x, gy, gw, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, off_d, off_h, off_w, 7u, stream);
}

/* kd_mask: bit kd set = the depth taps whose gradients are computed (the others stay zero) -- 2 for maps stacked as the planes
 * of one volume (2D convolutions: only the middle depth slice exists).  Cin = 8: 8-channel rows of x on the K = 16 kernel (TMA
 * zero fill), gw is then [27][16][cout] with rows 8..15 zero. */
extern "C" int mvsb200_conv3d_s1_wgrad_ex(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Cin, int Do,
                                          int Ho, int Wo, int cout, int off_d, int off_h, int off_w, unsigned kd_mask, void* stream) {
    MVS_REQUIRE(x && gy && gw, "conv3d_s1_wgrad: null pointer");
    MVS_REQUIRE(kd_mask >= 1u && kd_mask <= 7u, "conv3d_s1_wgrad: depth-tap mask %u", kd_mask);
    const int cin_real = Cin;
    if (Cin == 8) Cin = 16;
    MVS_REQUIRE(aligned16(x) && aligned16(gy) && aligned16(gw), "conv3d_s1_wgrad: pointers must be 16-byte aligned");
    MVS_REQUIRE(B >= 1 && Di >= 1 && Hi >= 1 && Wi >= 1 && Do >= 1 && Ho >= 1 && Wo >= 1, "conv3d_s1_wgrad: bad shape");
    MVS_REQUIRE(cout == 8 || cout == 16 || cout == 32 || cout == 64, "conv3d_s1_wgrad: cout must be 8, 16, 32 or 64 (got %d)", cout);
    cudaStream_t st = (cudaStream_t)stream;
    MVS_CUDA(cudaMemsetAsync(gw, 0, (size_t)27 * Cin * cout * sizeof(float), st));
    // gy channels per launch: (depth taps) x (1 or 2 kw blocks) x (kh, co) columns must fit the 512 TMEM columns.  64-channel x
    // (two kw blocks): 32 gy channels fit only with ONE depth tap per launch (2 x 96 columns) -- three launches per channel
    // chunk, each at twice the MMA N extent, instead of one at 16 channels: the A operand (the x slab, 4 KB per MMA) is read
    // from shared memory half as often per flop (measured: conv_3_1 1.03 -> see profiles/r02_k3_notes.md)
    if (Cin == 64 && cout % 32 == 0 && cout <= 64) {
        // ONE launch: the (channel chunk, depth tap) combinations are roles of neighbouring CTAs that walk the items together
        // (the six launches of the earlier form each read x and gy from DRAM)
        int role_co0[8], role_kd[8], n_roles = 0;
        for (int co0 = 0; co0 < cout; co0 += 32)
            for (int kd = 0; kd < 3; ++kd) { role_co0[n_roles] = co0; role_kd[n_roles] = 1 << kd; ++n_roles; }
        for (int r = 0; r < n_roles;) {                                     // roles of depth taps that are masked out do nothing: drop them
            if (role_kd[r] & (int)kd_mask) { ++r; continue; }
            for (int q = r; q + 1 < n_roles; ++q) { role_co0[q] = role_co0[q + 1]; role_kd[q] = role_kd[q + 1]; }
            --n_roles;
        }
        return launch_wgrad<64, 32>(x, gy, gw, B, Di, Hi, Wi, Do, Ho, Wo, cout, 0, off_d, off_h, off_w, st, 1, 0, 0, 0, 1u, nullptr, n_roles,
                                    role_co0, role_kd);
    }
    const int nco_max = Cin == 64 ? 16 : 32;
    const int nco = cout < nco_max ? cout : nco_max;
    for (int co0 = 0; co0 < cout; co0 += nco) {
        int rc = MVSB200_OK;
        if (!dispatch(WgradChannels{}, Cin, nco, rc, [&](auto c) {
                using C = decltype(c);
                return launch_wgrad<C::k, C::n>(x, gy, gw, B, Di, Hi, Wi, Do, Ho, Wo, cout, co0, off_d, off_h, off_w, st, 1, 0, 0, 0,
                                                kd_mask, nullptr, 1, nullptr, nullptr, cin_real);
            }))
            MVS_FAIL(MVSB200_E_UNSUPPORTED, "conv3d_s1_wgrad: unsupported channels Cin=%d cout=%d", Cin, cout);
        MVS_TRY(rc);
    }
    return MVSB200_OK;
}

// the stride-2 forward in launches of up to 64 filter rows.  stats: null, or the workspace of mvsb200_conv3d_s2_fwd_stats,
// whose rows the launches' epilogues fill; the largest grid of the launches is then raised into *n_blocks.
static int conv3d_s2_fwd_rows(const void* x, const void* w_packed, void* y, int B, int Dx, int Hx, int Wx, int Cin, int Do, int Ho,
                              int Wo, int cout, int y_cs, int n_rows, int pad_d, int pad_h, int pad_w, float* stats, int* n_blocks,
                              cudaStream_t st) {
    const char* name = "conv3d_s2_fwd";
    MVS_TRY(check_pointers(name, {x, w_packed, y}));
    MVS_REQUIRE(B >= 1 && Dx >= 1 && Hx >= 2 && Wx >= 2 && Do >= 1 && Ho >= 1 && Wo >= 1, "%s: bad shape", name);
    MVS_REQUIRE(cout >= 8 && cout % 8 == 0 && cout <= n_rows && n_rows % 16 == 0 && n_rows <= 128, "%s: cout %d / n_rows %d", name, cout,
                n_rows);
    MVS_REQUIRE(y_cs >= cout && y_cs % 8 == 0, "%s: output channel stride %d", name, y_cs);
    MVS_TRY(check_pads(name, pad_d, pad_h, pad_w));
    // filter rows per launch: up to 64 (27 x 64 x Cin taps resident in shared memory), then 48 / 32 / 16
    for (int row0 = 0; row0 < n_rows && row0 < cout;) {
        const int left = n_rows - row0;
        const int nmax = Cin == 64 ? 32 : 64;
        const int nout = left >= nmax ? nmax : left;
        const int c_here = cout - row0 < nout ? cout - row0 : nout;
        int rc = MVSB200_OK;
        if (!dispatch(S2Channels{}, Cin, nout, rc, [&](auto c) {
                using C = decltype(c);
                return launch_conv_s2<C::k, C::n>(x, w_packed, y, B, Dx, Hx, Wx, Do, Ho, Wo, c_here, y_cs, row0, n_rows, row0, pad_d,
                                                  pad_h, pad_w, st, Cin, stats, cout, n_blocks);
            }))
            MVS_FAIL(MVSB200_E_UNSUPPORTED, "%s: unsupported channels Cin=%d rows=%d", name, Cin, nout);
        MVS_TRY(rc);
        row0 += nout;
    }
    return MVSB200_OK;
}

extern "C" int mvsb200_conv3d_s2_fwd(const void* x, const void* w_packed, void* y, int B, int Dx, int Hx, int Wx, int Cin, int Do,
                                     int Ho, int Wo, int cout, int y_cs, int n_rows, int pad_d, int pad_h, int pad_w, void* stream) {
    return conv3d_s2_fwd_rows(x, w_packed, y, B, Dx, Hx, Wx, Cin, Do, Ho, Wo, cout, y_cs, n_rows, pad_d, pad_h, pad_w, nullptr, nullptr,
                              (cudaStream_t)stream);
}

/* mvsb200_conv3d_s2_fwd that also leaves sums[2][cout] = (sum, sum of squares) of its outputs per channel, accumulated in the
 * kernels' epilogues (fp32 accumulators) and combined in fixed order: the box BatchNorm that follows needs no statistics pass.
 * workspace: at least (SM count) * 2 * cout floats. */
extern "C" int mvsb200_conv3d_s2_fwd_stats(const void* x, const void* w_packed, void* y, int B, int Dx, int Hx, int Wx, int Cin, int Do,
                                           int Ho, int Wo, int cout, int y_cs, int n_rows, int pad_d, int pad_h, int pad_w,
                                           float* workspace, float* sums, void* stream) {
    MVS_REQUIRE(workspace && sums, "conv3d_s2_fwd_stats: null statistics buffers");
    cudaStream_t st = (cudaStream_t)stream;
    MVS_CUDA(cudaMemsetAsync(workspace, 0, (size_t)sm_count() * 2 * cout * sizeof(float), st));      // launches may differ in grid size
    int n_blocks = 0;
    MVS_TRY(conv3d_s2_fwd_rows(x, w_packed, y, B, Dx, Hx, Wx, Cin, Do, Ho, Wo, cout, y_cs, n_rows, pad_d, pad_h, pad_w, workspace,
                               &n_blocks, st));
    s2_stats_finalize_kernel<<<(2 * cout + 127) / 128, 128, 0, st>>>(workspace, n_blocks, cout, sums);
    MVS_CHECK_LAUNCH("s2_stats_finalize");
    return MVSB200_OK;
}

// one body for mvsb200_deconv3d_s2_fwd(_stats) (EPI = false: win, scale, shift and add null) and mvsb200_deconv3d_s2_fwd_affine
// (EPI = true, stats null; its caller has checked win, scale and shift for null)
template <bool EPI>
static int deconv3d_s2_fwd_body(const char* name, const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                const int64_t* y_strides4, float* stats, int* n_blocks_host, const int* win, const float* scale,
                                const float* shift, const void* add, void* stream) {
    MVS_TRY(check_pointers(name, {x, w_packed, y}, {y_strides4}));
    MVS_REQUIRE(add == nullptr || aligned16(add), "%s: pointers must be 16-byte aligned", name);
    MVS_REQUIRE(B >= 1 && B <= 65535 && Di >= 1 && Hi >= 1 && Wi >= 1 && Do >= 1 && Ho >= 1 && Wo >= 1, "%s: bad shape", name);
    MVS_REQUIRE(cout >= 8 && cout % 8 == 0 && cout <= n_rows && (n_rows == 16 || n_rows == 32),
                "%s: cout must be a multiple of 8 and n_rows 16 or 32 (cout=%d n_rows=%d)", name, cout, n_rows);
    MVS_TRY(check_pads(name, pad_d, pad_h, pad_w));
    if (EPI) {
        const int ext[3] = {Do, Ho, Wo};
        for (int a = 0; a < 3; ++a)
            MVS_REQUIRE(win[a] >= 0 && win[3 + a] >= 1 && win[a] + win[3 + a] <= ext[a],
                        "%s: window [%d, %d) outside the canvas extent %d (axis %d)", name, win[a], win[a] + win[3 + a], ext[a], a);
    }
    long long ys[4];
    MVS_TRY(copy_strides(name, y_strides4, ys));
    int rc = MVSB200_OK;
    if (!dispatch(ConvChannels{}, Cin, n_rows, rc, [&](auto c) {
            using C = decltype(c);
            return launch_deconv_s2<C::k, C::n, EPI>(x, w_packed, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, n_rows, pad_d, pad_h, pad_w, ys,
                                                     (cudaStream_t)stream, stats, n_blocks_host, win, scale, shift, add);
        }))
        MVS_FAIL(MVSB200_E_UNSUPPORTED, "%s: unsupported channels Cin=%d n_rows=%d", name, Cin, n_rows);
    return rc;
}

/* stats (may be NULL): [n_blocks][2][cout] fp32 per-CTA sums of the stored values and of their squares over the written canvas,
 * n_blocks returned through n_blocks_host (<= the device's SM count: size the buffer for that) -- the operand of
 * mvsb200_bn_finalize_affine, so the BatchNorm that follows a transposed convolution needs no statistics pass. */
extern "C" int mvsb200_deconv3d_s2_fwd_stats(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                             int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                             const int64_t* y_strides4, float* stats, int* n_blocks_host, void* stream) {
    return deconv3d_s2_fwd_body<false>("deconv3d_s2_fwd", x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, n_rows, pad_d, pad_h,
                                       pad_w, y_strides4, stats, n_blocks_host, nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int mvsb200_deconv3d_s2_fwd(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                       int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                       const int64_t* y_strides4, void* stream) {
    return mvsb200_deconv3d_s2_fwd_stats(x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, n_rows, pad_d, pad_h, pad_w, y_strides4,
                                         nullptr, nullptr, stream);
}

/* Eval-mode form of mvsb200_deconv3d_s2_fwd (include/mvs_b200.h): y = relu(acc * scale + shift) (+ add) on a window of the canvas
 * (deconv3d_s2_tc_kernel<.., EPI = true>). */
extern "C" int mvsb200_deconv3d_s2_fwd_affine(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                              int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                              const int* window6_host, const int64_t* y_strides4, const float* scale, const float* shift,
                                              const void* add, void* stream) {
    const char* name = "deconv3d_s2_fwd_affine";
    MVS_TRY(check_pointers(name, {}, {window6_host, scale, shift}));
    return deconv3d_s2_fwd_body<true>(name, x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, n_rows, pad_d, pad_h, pad_w,
                                      y_strides4, nullptr, nullptr, window6_host, scale, shift, add, stream);
}

/* Same convolution as mvsb200_conv3d_s1_fwd with the depth tap folded into the MMA N extent (conv3d_s1_kdn_kernel).
 * w_packed: [9 (kh,kw)][3 (kd)][n_rows][Cin] bf16.  planar: KdnParams::planar. */
template <bool AFF>
static int kdn_dispatch(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin, int Do, int Ho, int Wo,
                        int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w, int planar, void* stream, const char* name,
                        const float* scale, const float* shift) {
    MVS_TRY(check_s1_fwd(name, x, w_packed, y, B, Di, Hi, Wi, Do, Ho, Wo, cout, y_cs, n_rows));
    cudaStream_t st = (cudaStream_t)stream;
    for (int row0 = 0; row0 < n_rows && row0 < cout; row0 += 32) {
        const int nout = n_rows - row0 < 32 ? n_rows - row0 : 32;
        const int c_here = cout - row0 < nout ? cout - row0 : nout;
        int rc = MVSB200_OK;
        if (!dispatch(KdnChannels{}, Cin, nout, rc, [&](auto c) {
                using C = decltype(c);
                return launch_conv_kdn<C::k, C::n, AFF>(x, w_packed, y, B, Di, Hi, Wi, Do, Ho, Wo, c_here, y_cs, row0, n_rows, row0, off_d,
                                                        off_h, off_w, planar, st, Cin, scale, shift);
            }))
            MVS_FAIL(MVSB200_E_UNSUPPORTED, "%s: unsupported channels Cin=%d n_rows=%d", name, Cin, n_rows);
        MVS_TRY(rc);
    }
    return MVSB200_OK;
}

extern "C" int mvsb200_conv3d_s1_fwd_kdn(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                         int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                                         void* stream) {
    return kdn_dispatch<false>(x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, y_cs, n_rows, off_d, off_h, off_w, 0, stream,
                               "conv3d_s1_fwd_kdn", nullptr, nullptr);
}

/* 2D convolution 3x3 / padding 1 of N maps stacked as channel-last rows [N, H, W, Cin] -> [N, H, W, y_cs] (SURVEY §8 rows f1 / f2;
 * scripts/model.py:22-65, :129-152): conv3d_s1_kdn_kernel in its planar mode.  w_packed is the kdn operand [9 (kh,kw)][3][n_rows][Cin]
 * of which only the middle row block of every in-plane tap is read. */
extern "C" int mvsb200_conv2d_rows_fwd(const void* x, const void* w_packed, void* y, int N, int H, int W, int Cin, int cout, int y_cs,
                                       int n_rows, void* stream) {
    return kdn_dispatch<false>(x, w_packed, y, 1, N, H, W, Cin, N, H, W, cout, y_cs, n_rows, 0, -1, -1, 1, stream, "conv3d_s1_fwd_kdn",
                               nullptr, nullptr);
}

/* mvsb200_conv3d_s1_fwd_kdn (planar = 0) or mvsb200_conv2d_rows_fwd (planar = 1, B = 1, Di = Do = maps) with eval-mode BatchNorm +
 * ReLU in the epilogue: y = relu(acc * scale[c] + shift[c]), scale / shift fp32 [cout] device vectors. */
extern "C" int mvsb200_conv3d_s1_fwd_kdn_affine(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                                int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                                                int planar, const float* scale, const float* shift, void* stream) {
    const char* name = "conv3d_s1_fwd_kdn_affine";
    MVS_REQUIRE(scale && shift, "%s: null scale / shift", name);
    MVS_REQUIRE(planar == 0 || (planar == 1 && B == 1 && Di == Do && off_d == 0), "%s: planar mode takes B = 1, Di = Do, off_d = 0", name);
    return kdn_dispatch<true>(x, w_packed, y, B, Di, Hi, Wi, Cin, Do, Ho, Wo, cout, y_cs, n_rows, off_d, off_h, off_w, planar, stream, name,
                              scale, shift);
}

/* Weight gradient of the STRIDE-2 layers on the same kernel:  gw[k][cb][cs] = sum_o big(2o - pad + k)[cb] * small(o)[cs]
 * (per axis, k = 0..2, big zero outside its volume).  For a stride-2 convolution (model.py:104-110) big = its input, small =
 * the output gradient; for a stride-2 transposed convolution (model.py:115-121) big = the output gradient, small = its input
 * (gw then holds [k][Cout][Cin]).  Per output-parity class pi of (k - pad) the sum is a stride-1 correlation of the class's
 * sub-lattice of `big` (a TMA map with doubled strides) with `small`; each class launch issues only the depth taps it needs
 * and drops the in-plane taps of other classes. */
extern "C" int mvsb200_conv3d_s2_wgrad(const void* big, const void* small, float* gw, int B, int Db, int Hb, int Wb, int Cb,
                                       int Ds, int Hs, int Ws, int Cs, int pad_d, int pad_h, int pad_w, void* stream) {
    const char* name = "conv3d_s2_wgrad";
    MVS_TRY(check_pointers(name, {big, small, gw}));
    MVS_REQUIRE(B >= 1 && Db >= 1 && Hb >= 1 && Wb >= 1 && Ds >= 1 && Hs >= 1 && Ws >= 1, "%s: bad shape", name);
    MVS_REQUIRE(Cb == 16 || Cb == 32 || Cb == 64, "%s: the strided operand must have 16, 32 or 64 channels (got %d)", name, Cb);
    MVS_REQUIRE(Cs >= 8 && Cs % 8 == 0, "%s: the dense operand needs a multiple of 8 channels (got %d)", name, Cs);
    MVS_TRY(check_pads(name, pad_d, pad_h, pad_w));
    cudaStream_t st = (cudaStream_t)stream;
    MVS_CUDA(cudaMemsetAsync(gw, 0, (size_t)27 * Cb * Cs * sizeof(float), st));
    const int pads[3] = {pad_d, pad_h, pad_w};
    const int nb[3] = {Db, Hb, Wb};
    const int nco_max = Cb == 64 ? 16 : 32;
    for (int c = 0; c < 8; ++c) {
        const int par[3] = {c >> 2 & 1, c >> 1 & 1, c & 1};
        int sub[3];
        bool empty = false;
        for (int ax = 0; ax < 3; ++ax) { sub[ax] = (nb[ax] - par[ax] + 1) / 2; if (sub[ax] < 1) empty = true; }
        if (empty) continue;
        // filter taps of this class per axis: k with (k - pad - par) even; shift s = (k - pad - par)/2 in {-1, 0}; kernel tap t = s + 1
        int tap_map[27];
        for (int t = 0; t < 27; ++t) tap_map[t] = -1;
        unsigned kd_mask = 0;
        int n_taps = 0;
        for (int kd = 0; kd < 3; ++kd)
            for (int kh = 0; kh < 3; ++kh)
                for (int kw = 0; kw < 3; ++kw) {
                    const int k[3] = {kd, kh, kw};
                    int t[3];
                    bool ok = true;
                    for (int ax = 0; ax < 3; ++ax) {
                        const int v = k[ax] - pads[ax] - par[ax];
                        if (v & 1) { ok = false; break; }
                        t[ax] = v / 2 + 1;                   // v is even and <= 0: exact
                        if (t[ax] < 0 || t[ax] > 2) { ok = false; break; }
                    }
                    if (!ok) continue;
                    tap_map[(t[0] * 3 + t[1]) * 3 + t[2]] = (kd * 3 + kh) * 3 + kw;
                    kd_mask |= 1u << t[0];
                    ++n_taps;
                }
        if (n_taps == 0) continue;
        const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(big) + (((size_t)par[0] * Hb + par[1]) * Wb + par[2]) * Cb;
        for (int co0 = 0; co0 < Cs;) {
            const int left = Cs - co0;
            const int nco = left >= nco_max ? nco_max : (left >= 16 ? 16 : 8);
            int rc = MVSB200_OK;
            if (!dispatch(WgradChannels{}, Cb, nco, rc, [&](auto c) {
                    using C = decltype(c);
                    return launch_wgrad<C::k, C::n>(base, small, gw, B, sub[0], sub[1], sub[2], Ds, Hs, Ws, Cs, co0, -1, -1, -1, st, 2, Db,
                                                    Hb, Wb, kd_mask, tap_map);
                }))
                MVS_FAIL(MVSB200_E_UNSUPPORTED, "%s: unsupported channels %d / %d", name, Cb, nco);
            MVS_TRY(rc);
            co0 += nco;
        }
    }
    return MVSB200_OK;
}
