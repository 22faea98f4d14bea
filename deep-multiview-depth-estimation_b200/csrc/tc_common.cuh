// tcgen05 / TMA / mbarrier PTX wrappers, UMMA shared-memory descriptors, the tensor-map encoder and the host-side launch
// helpers shared by the tensor-core convolution kernels of libmvs_b200.so (conv3d_tc.cu, conv3d_s2_bwd.cu).  sm_100a only.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <initializer_list>

namespace {

// ---- PTX wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3,
                                            int c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
                 : "memory");
}
// one lane of a converged warp (the form the compiler recognises as single-thread issue: no uniformisation loops
// around the tcgen05 / TMA instructions it guards)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .b32 rx;\n\t.reg .pred px;\n\t"
        "elect.sync rx|px, 0xffffffff;\n\t"
        "@px mov.s32 %0, 1;\n\t}"
        : "+r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
        "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
template <int N>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, uint32_t (&v)[N]);
template <>
__device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                   "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
}
template <>
__device__ __forceinline__ void tmem_ld<32>(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,"
        "%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
          "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
          "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
          "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory descriptor of a K-major operand whose rows are ROWB bytes (= the swizzle span) apart.
// Measured on B200 (tools/test_conv_tc.py, round 1): the hardware applies the swizzle XOR to the ABSOLUTE shared-memory
// address, exactly as TMA does when it writes the tile, so a start address shifted by any number of voxel rows (not
// only by whole 8-row swizzle atoms) addresses the shifted operand correctly with the base-offset field left 0.
// (Setting base_offset = (addr >> 7) & 7 for unaligned starts gives wrong results.)
template <int ROWB>
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
    constexpr uint64_t layout = ROWB == 128 ? 2 : (ROWB == 64 ? 4 : 6);          // SWIZZLE_128B / 64B / 32B
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;                                                       // LBO: unused for swizzled K-major
    d |= (uint64_t)((8 * ROWB) >> 4) << 32;                                       // SBO: 8 rows
    d |= (uint64_t)1 << 46;                                                       // descriptor version (Blackwell)
    d |= layout << 61;
    return d;
}

// one tcgen05.mma, descriptors given as (lo, hi) halves so the issue loop only does 32-bit adds on the start address
__device__ __forceinline__ void umma_bf16_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                               uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}" ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi),
        "r"(idesc), "r"(accumulate)
        : "memory");
}

// MN-major operand descriptor: rows (K) are ROWB bytes apart (= one swizzle atom of channels), MN atoms `atom_stride`
// bytes apart
template <int ROWB>
__device__ __forceinline__ uint64_t umma_desc_mn(uint32_t saddr, uint32_t atom_stride) {
    constexpr uint64_t layout = ROWB == 128 ? 2 : (ROWB == 64 ? 4 : (ROWB == 32 ? 6 : 0));
    uint64_t d = (uint64_t)((saddr >> 4) & 0x3fff);
    if (ROWB == 16) {
        d |= (uint64_t)(128 >> 4) << 16;                      // no swizzle: LBO = stride between 8-row K groups
        d |= (uint64_t)((atom_stride >> 4) & 0x3fff) << 32;   //             SBO = stride between 8-channel MN atoms
    } else {
        d |= (uint64_t)((atom_stride >> 4) & 0x3fff) << 16;   // LBO = stride between MN atoms
        d |= (uint64_t)((8 * ROWB) >> 4) << 32;               // SBO = stride between 8-row K groups
    }
    d |= (uint64_t)1 << 46;
    d |= layout << 61;
    return d;
}

// ---- host side ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// swizzle of a box whose rows are rowb bytes (one swizzle span); 16-byte rows are not swizzled
CUtensorMapSwizzle swizzle_for(int rowb) {
    return rowb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                       : (rowb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : (rowb == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE));
}

// bf16 tensor map of `rank` dims (innermost first), rank - 1 byte strides and a box in elements; L2 128-byte promotion,
// elements outside the tensor read as zeros.  Errors name the launcher and the operand: `what`, followed by `index` if it
// is not negative.
int encode_tiled(CUtensorMap* map, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides,
                 const cuuint32_t* box, CUtensorMapSwizzle swizzle, const char* name, const char* what, int index = -1) {
    EncodeTiledFn enc = encode_fn();
    MVS_REQUIRE(enc != nullptr, "%s: cuTensorMapEncodeTiled is not available from the driver", name);
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS && index >= 0) MVS_FAIL(MVSB200_E_BADARG, "%s: cuTensorMapEncodeTiled(%s %d) failed (%d)", name, what, index, (int)r);
    MVS_REQUIRE(r == CUDA_SUCCESS, "%s: cuTensorMapEncodeTiled(%s) failed (%d)", name, what, (int)r);
    return MVSB200_OK;
}

// dense channel-last volume [B][D][H][W][C] read in boxes of box_c channels x box_w voxels x box_h lines of one plane (a box
// wider than C reads the missing channels as zeros)
int encode_volume(CUtensorMap* map, const void* base, int C, int box_c, int W, int H, int D, int B, int box_w, int box_h,
                  const char* name, const char* what, int index = -1) {
    const cuuint64_t row = (cuuint64_t)C * 2;
    const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
    const cuuint64_t strides[4] = {row, row * W, row * W * H, row * W * H * D};
    const cuuint32_t box[5] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1, 1};
    return encode_tiled(map, base, 5, dims, strides, box, swizzle_for(2 * box_c), name, what, index);
}

// packed filter: `rows` rows of C channels, read box_rows rows at a time
int encode_filter(CUtensorMap* map, const void* base, int C, int rows, int box_rows, const char* name, const char* what,
                  int index = -1) {
    const cuuint64_t dims[2] = {(cuuint64_t)C, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {(cuuint64_t)C * 2};
    const cuuint32_t box[2] = {(cuuint32_t)C, (cuuint32_t)box_rows};
    return encode_tiled(map, base, 2, dims, strides, box, swizzle_for(2 * C), name, what, index);
}

// Split `extent` planes (or lines) into runs for persistent CTAs: `walkers` CTAs take the tiles * runs * B items in turn and
// an item costs its run length + `overhead` (halo planes, pipeline fill).  Picks the run count with the least
// (items per walker) x (cost per item); a run count that would leave a run empty is skipped.
struct Runs { int nchunks, chunk; };
Runs choose_runs(long tiles, int B, int extent, long walkers, int overhead) {
    long best_cost = -1;
    int best = 1;
    for (int nc = 1; nc <= extent; ++nc) {
        const int dc = (extent + nc - 1) / nc;
        if ((long)(nc - 1) * dc >= extent) continue;
        const long items = tiles * nc * B;
        const long cost = ((items + walkers - 1) / walkers) * (dc + overhead);
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = nc; }
    }
    return Runs{best, (extent + best - 1) / best};
}

// argument checks shared by the convolution entry points; `name` starts the message.  Pointers in `aligned` must be
// non-null and 16-byte aligned, those in `present` non-null.
int check_pointers(const char* name, std::initializer_list<const void*> aligned, std::initializer_list<const void*> present = {}) {
    for (const void* p : aligned) MVS_REQUIRE(p, "%s: null pointer", name);
    for (const void* p : present) MVS_REQUIRE(p, "%s: null pointer", name);
    for (const void* p : aligned) MVS_REQUIRE(::mvsb200::aligned16(p), "%s: pointers must be 16-byte aligned", name);
    return MVSB200_OK;
}
int check_pads(const char* name, int pad_d, int pad_h, int pad_w) {
    MVS_REQUIRE(pad_d >= 1 && pad_d <= 2 && pad_h >= 1 && pad_h <= 2 && pad_w >= 1 && pad_w <= 2, "%s: pad must be 1 or 2 per axis", name);
    return MVSB200_OK;
}
// output voxel-row strides (b, d, h, w) in elements, each a multiple of 8
int copy_strides(const char* name, const int64_t* s, long long ys[4]) {
    for (int i = 0; i < 4; ++i) {
        ys[i] = (long long)s[i];
        MVS_REQUIRE(ys[i] % 8 == 0, "%s: output strides must be multiples of 8 elements", name);
    }
    return MVSB200_OK;
}

// 32-byte global loads / stores (sm_100: ld/st.global.v8.b32): one instruction per 16-channel bf16 piece of a voxel row
struct U8 { uint32_t v[8]; };
__device__ __forceinline__ U8 ld_u8(const void* p) {
    U8 r;
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7]) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_u8(void* p, const U8& r) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(r.v[0]), "r"(r.v[1]), "r"(r.v[2]), "r"(r.v[3]),
                 "r"(r.v[4]), "r"(r.v[5]), "r"(r.v[6]), "r"(r.v[7]) : "memory");
}


// ---- stride-2 transposed convolution: the 27 (output-parity class, filter tap) pairs ---------------------------------
//   out[2J + par] = sum over the filter taps k with (par + pad - k) even of W[k] . in[J + (par + pad - k)/2]   (per axis)
// Slab tap t = (par + pad - k)/2 + 1 per axis (input index J + t - 1); for pad in {1, 2} only t = 1, 2 occur.  Classes that
// read the same INPUT SHIFT (td,th,tw) share the A operand of the MMA.  The table below arranges the pairs for ONE MMA PER
// INPUT SHIFT.  Per axis one output parity reads both input shifts (bit
// u = 1) and the other only the main one; the 8 classes are placed in Gray-code order of (u_d, u_h, u_w), so the classes that
// read a given shift occupy a short RANGE of accumulator blocks -- the MMA of the shift covers the whole range, blocks of
// classes that do not read the shift get an all-zero filter slot (tap index 27 of the packed weights).  8 MMAs per K step
// instead of 14: on the shared-memory operand-feed roof an MMA costs its 4 KB A read whatever its N, so fewer, wider MMAs win.
struct DeconvWide {
    int tap_k[40];                  // filter tap held by shared-memory slot e; 27 = the all-zero tap
    int n_slots;
    int n_groups;                   // <= 8
    int grp_td[8], grp_th[8], grp_tw[8];      // input shift (slab tap per axis, 1 or 2)
    int grp_pos0[8], grp_npos[8];             // first accumulator block and number of adjacent blocks the MMA covers
    int grp_slot0[8];
    int grp_first[8];                         // 1: initialises its accumulators (covers all 8 blocks)
    int cls_of_pos[8];              // output-parity class (pd*4 + ph*2 + pw) of accumulator block pos
};

inline int build_deconv_wide(int pad_d, int pad_h, int pad_w, int NOUT, DeconvWide& p) {
    const int pads[3] = {pad_d, pad_h, pad_w};
    // per axis: taps of a parity -> (k, t); the parity with two taps has u = 1
    int two[3];                                          // parity that reads both shifts
    for (int ax = 0; ax < 3; ++ax) {
        int cnt[2] = {0, 0};
        for (int par = 0; par < 2; ++par)
            for (int k = 0; k < 3; ++k) {
                const int v = par + pads[ax] - k;
                if (v & 1) continue;
                const int t = v / 2 + 1;
                MVS_REQUIRE(t >= 1 && t <= 2, "deconv3d_s2: padding %d gives an input shift outside {0, +1}", pads[ax]);
                ++cnt[par];
            }
        MVS_REQUIRE(cnt[0] + cnt[1] == 3 && (cnt[0] == 2 || cnt[1] == 2), "deconv3d_s2: padding %d does not split the 3 taps 2 + 1", pads[ax]);
        two[ax] = cnt[1] == 2 ? 1 : 0;
    }
    static const int gray[8] = {0, 1, 3, 2, 6, 7, 5, 4};     // position -> (u_d u_h u_w) as a 3-bit number
    int pos_of_cls[8];
    for (int pos = 0; pos < 8; ++pos) {
        const int u[3] = {gray[pos] >> 2 & 1, gray[pos] >> 1 & 1, gray[pos] & 1};
        int par[3];
        for (int ax = 0; ax < 3; ++ax) par[ax] = u[ax] ? two[ax] : 1 - two[ax];
        p.cls_of_pos[pos] = par[0] * 4 + par[1] * 2 + par[2];
        pos_of_cls[p.cls_of_pos[pos]] = pos;
    }
    int pair_k[8][27];                                   // pair_k[pos][shift] = filter tap or -1
    for (int c = 0; c < 8; ++c)
        for (int t = 0; t < 27; ++t) pair_k[c][t] = -1;
    for (int c = 0; c < 8; ++c) {
        const int par[3] = {c >> 2 & 1, c >> 1 & 1, c & 1};
        for (int kd = 0; kd < 3; ++kd)
            for (int kh = 0; kh < 3; ++kh)
                for (int kw = 0; kw < 3; ++kw) {
                    const int k[3] = {kd, kh, kw};
                    int t[3];
                    bool ok = true;
                    for (int ax = 0; ax < 3; ++ax) {
                        const int v = par[ax] + pads[ax] - k[ax];
                        if (v & 1) { ok = false; break; }
                        t[ax] = v / 2 + 1;
                    }
                    if (ok) pair_k[pos_of_cls[c]][(t[0] * 3 + t[1]) * 3 + t[2]] = (kd * 3 + kh) * 3 + kw;
                }
    }
    int order[27], users[27];
    for (int t = 0; t < 27; ++t) {
        order[t] = t;
        users[t] = 0;
        for (int c = 0; c < 8; ++c) users[t] += pair_k[c][t] >= 0;
    }
    for (int i = 0; i < 27; ++i)
        for (int j = i + 1; j < 27; ++j)
            if (users[order[j]] > users[order[i]]) { const int tmp = order[i]; order[i] = order[j]; order[j] = tmp; }
    int ng = 0, slot = 0;
    for (int oi = 0; oi < 27; ++oi) {
        const int t = order[oi];
        if (users[t] == 0) continue;
        int lo = 8, hi = -1;
        for (int c = 0; c < 8; ++c)
            if (pair_k[c][t] >= 0) { lo = c < lo ? c : lo; hi = c > hi ? c : hi; }
        MVS_REQUIRE(ng < 8 && slot + (hi - lo + 1) <= 40 && (hi - lo + 1) * NOUT <= 256, "deconv3d_s2: wide group table overflow");
        MVS_REQUIRE(ng > 0 || (lo == 0 && hi == 7), "deconv3d_s2: the first shift does not reach every class");
        p.grp_td[ng] = t / 9; p.grp_th[ng] = t / 3 % 3; p.grp_tw[ng] = t % 3;
        p.grp_pos0[ng] = lo; p.grp_npos[ng] = hi - lo + 1; p.grp_slot0[ng] = slot; p.grp_first[ng] = ng == 0 ? 1 : 0;
        for (int c = lo; c <= hi; ++c) p.tap_k[slot++] = pair_k[c][t] >= 0 ? pair_k[c][t] : 27;
        ++ng;
    }
    p.n_groups = ng;
    p.n_slots = slot;
    for (int g = ng; g < 8; ++g) { p.grp_td[g] = p.grp_th[g] = p.grp_tw[g] = 1; p.grp_pos0[g] = p.grp_npos[g] = p.grp_slot0[g] = p.grp_first[g] = 0; }
    for (int e = slot; e < 40; ++e) p.tap_k[e] = 27;
    return MVSB200_OK;
}

}  // namespace
