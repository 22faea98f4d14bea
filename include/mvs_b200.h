/*
 * mvs_b200.h  --  C ABI of libmvs_b200.so, the sm_100a implementation of MVSNet's plane-sweep
 * hot path (homography warp -> variance cost volume -> 3D-conv regulariser -> softmax + depth).
 *
 * Drop-in boundary.  The reference (bcollico/Deep-Multiview-Depth-Estimation) is pure Python: its
 * "FFI" for this path is the set of Python callables that scripts/model.py:5-7 imports by name.
 * Each entry point below cites the reference interface it sits under; INTEGRATION.md shows the
 * ctypes binding and the 3-line swap a maintainer adds.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - return value: 0 on success, <0 on error (MVSB200_E_*); mvsb200_last_error() gives the
 *     message for the calling thread.  No entry point synchronises the device.
 *   - the caller owns and allocates every buffer; nothing is retained after return.
 *   - thread-safe for concurrent calls on distinct streams.
 *
 * Volume layout ("plane-major, channel-last"): a volume with logical shape [B, C, D, h, w] is stored
 * as B x D x h x w x C, i.e. torch's channels_last_3d strides.  A voxel (b,d,y,x) is one contiguous
 * row of C values (128 B fp32 / 64 B bf16 at C = 32).  Feature maps [N, C, h, w] are stored
 * N x h x w x C (torch channels_last).
 */
#ifndef MVS_B200_H_
#define MVS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVSB200_ABI_VERSION 1

#define MVSB200_OK             0
#define MVSB200_E_BADARG      -1   /* unsupported shape / null pointer / misaligned pointer */
#define MVSB200_E_LAUNCH      -2   /* CUDA launch or runtime failure */
#define MVSB200_E_UNSUPPORTED -3   /* valid request this build does not cover */

#define MVSB200_F32  0
#define MVSB200_BF16 1

/* Floats per view in the `view_params` table of the warp kernels.
 *   [0..8]  A'  = S * A^-1, row major          (S = diag(w/(w-1), h/(h-1), 1), kornia's resample)
 *   [9..11] g'  = S * A^-1 u
 *   [12..14] r  = w^T A^-1
 *   [15]    reserved (0)
 * with H_i(d) = A - u w^T / d the matrix of scripts/homography.py:61-75, so that the sampling
 * position of destination pixel p = (x,y,1) on plane d is
 *   q = A' p + g' (r.p) * tinv[i][d],   ix = qx/qz - 0.5,  iy = qy/qz - 0.5,
 *   tinv[i][d] = 1 / (depth_i[d] - w^T A^-1 u)            (NaN marks a d == 0 plane: output NaN,
 *                                                          as the reference's division by d does) */
#define MVSB200_VIEW_PARAM_FLOATS 16

int         mvsb200_abi_version(void);
const char* mvsb200_last_error(void);
/* number of kernel launches issued through this library by the calling process (all threads) */
uint64_t    mvsb200_launch_count(void);

/* ---- layout helpers --------------------------------------------------------------------------
 * FeatureEncoder output (scripts/model.py:174) is NCHW; the warp kernels read channel-last rows. */
int mvsb200_nchw_to_nhwc_f32(const float* src, float* dst, int N, int C, int H, int W, void* stream);
int mvsb200_nhwc_to_nchw_f32(const float* src, float* dst, int N, int C, int H, int W, void* stream);

/* ---- K1: fused homography warp + variance cost volume -------------------------------------------
 * Replaces homography_warping's plane loop + kornia.warp_perspective (scripts/homography.py:78-90)
 * AND assemble_cost_volume (scripts/costvolume.py:3-16) in one pass; the N warped volumes are never
 * written.  feat: [B*V, h, w, C] fp32, view index b*V+v with v = 0 the reference view.
 * view_params: [B*V, 16] fp32, tinv: [B*V, D] fp32.  cost: [B, D, h, w, C] of cost_dtype.
 * Supported: C == 32, 2 <= V <= 8. */
int mvsb200_warp_variance_fwd(const float* feat, const float* view_params, const float* tinv,
                              void* cost, int cost_dtype,
                              int B, int V, int C, int D, int h, int w, void* stream);

/* ---- K2: backward of K1 wrt the feature maps -----------------------------------------------------
 * The gradient the reference obtains by autograd through grid_sample and the variance
 * (scripts/homography.py:85-90, scripts/costvolume.py:10-14).  gcost: [B, D, h, w, C] of
 * gcost_dtype.  gfeat: [B*V, h, w, C] fp32, ZEROED BY THIS CALL, then accumulated. */
int mvsb200_warp_variance_bwd(const float* feat, const float* view_params, const float* tinv,
                              const void* gcost, int gcost_dtype, float* gfeat,
                              int B, int V, int C, int D, int h, int w, void* stream);

/* ---- parity/debug: materialise the warped volumes exactly as homography_warping returns them ----
 * warped: [B*V, C, D, h, w] fp32, plain contiguous NCDHW (scripts/homography.py:92). */
int mvsb200_warp_materialize(const float* feat, const float* view_params, const float* tinv,
                             float* warped, int B, int V, int C, int D, int h, int w, void* stream);

/* ---- assemble_cost_volume on a plain, already materialised tensor (scripts/costvolume.py:3-16) ---
 * x: [B, V, M] fp32 (M = C*D*h*w), out: [B, M].  Backward: gx = (2/V)(x - mean) * gout. */
int mvsb200_variance_views_fwd(const float* x, float* out, int B, int V, int64_t M, void* stream);
int mvsb200_variance_views_bwd(const float* x, const float* gout, float* gx, int B, int V, int64_t M, void* stream);

/* ---- K4: depth-axis softmax + "top-N" expected depth ----------------------------------------------
 * Replaces CostVolumeReg.Norm = Softmax(dim=2) (scripts/model.py:96,123) and extract_depth_map
 * (scripts/depthmap.py:4-22).  in: [B, D, h, w] fp32 (logits if apply_softmax, else probabilities).
 * prob (out, may be NULL when !apply_softmax): [B, D, h, w].  depths: [B, D] fp32 or NULL.
 * ranks (out, may be NULL): [B, n_keep, h, w] int32, n_keep = min(n_est, D): position of plane j in
 * the stable descending sort over D == the planes the reference keeps.  depth (out, NULL iff depths
 * is NULL): [B, h, w].  D <= 1024. */
int mvsb200_softmax_depth_fwd(const float* in, int apply_softmax, const float* depths,
                              float* prob, int32_t* ranks, float* depth,
                              int B, int D, int h, int w, int n_est, void* stream);

/* mvsb200_softmax_depth_fwd that also writes conf [B, h, w] (required, as are depths and depth): MVSNet's photometric
 * confidence, the probability mass of the planes k0-1 .. k0+2 (clipped to [0, D-1]) where k0 = floor((depth - d_0) / (d_1 - d_0)),
 * summed in ascending k in fp32; 1 when D == 1; NaN for a non-finite depth or summed probability.  prob, ranks and depth are
 * bit-identical to mvsb200_softmax_depth_fwd. */
int mvsb200_softmax_depth_conf_fwd(const float* in, int apply_softmax, const float* depths,
                                   float* prob, int32_t* ranks, float* depth, float* conf,
                                   int B, int D, int h, int w, int n_est, void* stream);

/* the same confidence from a probability volume prob [B, D, h, w] and depth map [B, h, w] that already exist; bit-identical to the
 * conf of mvsb200_softmax_depth_conf_fwd on the same values */
int mvsb200_depth_confidence(const float* prob, const float* depth, const float* depths, float* conf,
                             int B, int D, int h, int w, void* stream);

/* depth from precomputed ranks (the cheap second half when softmax ran earlier, in CostVolumeReg) */
int mvsb200_depth_from_ranks(const float* prob, const int32_t* ranks, const float* depths, float* depth,
                             int B, int D, int h, int w, int n_keep, void* stream);

/* d depth / d prob: dense [B, D, h, w] with n_keep non-zeros per pixel (mask is constant, as in autograd
 * through scripts/depthmap.py:12-19).  gprob is fully written. */
int mvsb200_depth_bwd(const float* prob, const int32_t* ranks, const float* depths, const float* gdepth,
                      float* gprob, int B, int D, int h, int w, int n_keep, void* stream);

/* softmax backward over D: glogits = prob * (gprob - sum_D(gprob * prob)) */
int mvsb200_softmax_bwd(const float* prob, const float* gprob, float* glogits,
                        int B, int D, int h, int w, void* stream);

/* ---- K3: 3x3x3 stride-1 convolution, implicit GEMM on tcgen05 tensor cores fed by TMA ---------------
 * Replaces nn.Conv3d(k=3, stride=1, bias=False) of CostVolumeReg (scripts/model.py:223-234; the layers
 * conv_0_0, conv_1_1, conv_2_1, conv_3_1 at :101-113) and, with the flipped/transposed filter, autograd's
 * data gradient of the same layers.  bf16 in, fp32 accumulate (TMEM), bf16 out.
 *   x        [B, Di, Hi, Wi, Cin]  bf16, dense (channels_last_3d of a [B,Cin,Di,Hi,Wi] volume), Cin in {16,32,64}
 *   w_packed [27, n_rows, Cin]     bf16: tap-major (kd,kh,kw), then output channel (zero rows up to n_rows,
 *                                  n_rows in {16,32,64}), then input channel
 *   y        [B, Do, Ho, Wo, y_cs] bf16; channels [0, cout) of every voxel row are written (cout % 8 == 0)
 *   out(z,y,x) = sum_taps W[tap] . x(z + kd + off_d, y + kh + off_h, x + kw + off_w), zero outside the input:
 *   off = -1 is padding 1 (Do = Di), off = 0 a valid convolution (Do = Di - 2).
 */
int mvsb200_conv3d_s1_fwd(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                          int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                          void* stream);

/* Filter packing in one launch: the fp32 parameter w [dim0][dim1][3][3][3] of a Conv3d / ConvTranspose3d (scripts/model.py:223-234)
 * -> the bf16 [n_slots][n_rows][n_cols] K-major operand of the tensor-core kernels:
 *   out[s][r][c] = w[r*sr + (c + c0)*sc + taps[s]] for r < rows_real, c < cols_real, taps[s] >= 0; zero otherwise
 * (sr / sc: element strides of the row / column channel in w, i.e. 27*dim1 and 27 or the reverse; taps_host: HOST int array of
 * n_slots entries in 0..26 or -1 = an all-zero slot -- natural, flipped (data gradient), depth-innermost (kdn) orders). */
int mvsb200_pack_filter(const float* w, void* out, int n_slots, int n_rows, int n_cols, int rows_real, int cols_real,
                        int c0, int sr, int sc, const int* taps_host, void* stream);

/* [M, 8] bf16 voxel rows -> [M, 16] with channels 8..15 zero: operand of conv_0_0's data gradient (UMMA K = 16). */
int mvsb200_widen_rows_8to16_bf16(const void* src, void* dst, int64_t M, void* stream);

/* The same convolution with the depth tap folded into the MMA N extent (one MMA of N = 3*Cout per in-plane tap and K step,
 * running partial sums of the three contributing input planes in the epilogue's registers): 3x fewer A-operand reads from
 * shared memory.  w_packed: [9 (kh,kw)][3 (kd)][n_rows][Cin] bf16; everything else as mvsb200_conv3d_s1_fwd. */
int mvsb200_conv3d_s1_fwd_kdn(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                              int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                              void* stream);

/* mvsb200_conv3d_s1_fwd_kdn with eval-mode BatchNorm + ReLU in the epilogue: y = relu(acc * scale[c] + shift[c]) rounded once to
 * bf16, scale / shift fp32 [cout] device vectors (the filter stays unscaled: the same packed operand as the train path).
 * planar = 1: the 2D form of mvsb200_conv2d_rows_fwd (B = 1, Di = Do = number of maps, off_d = 0). */
int mvsb200_conv3d_s1_fwd_kdn_affine(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                     int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int off_d, int off_h, int off_w,
                                     int planar, const float* scale, const float* shift, void* stream);

/* Same kernel with a subset of the 27 taps (bit (kd*3+kh)*3+kw of tap_mask) and a strided output: the voxel row of
 * output (b,z,y,x) starts at y + b*ys[0] + z*ys[1] + y*ys[2] + x*ys[3] elements (y_strides4: HOST int64).  This is one
 * output-parity class of a stride-2 TRANSPOSED convolution (ConvTranspose3d, scripts/model.py:229-234, used at :115-121):
 * out[2j + par] = sum over the taps k with (par + p - k) even of W[k] . in[j + (par + p - k)/2]. */
int mvsb200_conv3d_s1_fwd_ex(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                             int Do, int Ho, int Wo, int cout, int n_rows, int off_d, int off_h, int off_w,
                             unsigned tap_mask, const int64_t* y_strides4_host, void* stream);

/* Weight gradient of the stride-2 layers (tcgen05, the stride-1 weight-gradient kernel on parity sub-lattices of the strided
 * operand):  gw[k][cb][cs] = sum_o big(2o - pad + k)[cb] * small(o)[cs], k = (kd,kh,kw), big zero outside its volume.
 *   stride-2 convolution (scripts/model.py:104-110):            big = input x [B,Db,Hb,Wb,Cb], small = output gradient
 *   stride-2 transposed convolution (scripts/model.py:115-121): big = output gradient, small = input (gw is [k][Cout][Cin])
 * big: bf16, Cb in {16,32,64}; small: bf16 [B,Ds,Hs,Ws,Cs], Cs % 8 == 0; gw: fp32 [27,Cb,Cs], zeroed by the call; pad in {1,2}. */
int mvsb200_conv3d_s2_wgrad(const void* big, const void* small, float* gw, int B, int Db, int Hb, int Wb, int Cb,
                            int Ds, int Hs, int Ws, int Cs, int pad_d, int pad_h, int pad_w, void* stream);

/* The same weight gradient in ONE launch (csrc/conv3d_s2_bwd.cu): lines of `big` are presented by TMA as rows of voxel PAIRS, so
 * a tcgen05.mma chain over a line accumulates the three kw taps of one (kd, kh) without any de-interleaved copy of `big`; a CTA
 * owns one depth tap and keeps its accumulators in TMEM over its whole run.  Replaces torch.nn.grad.conv3d_weight /
 * aten::convolution_backward for conv_{1,2,3}_0 (scripts/model.py:104-110; small = the 112 stacked output-gradient channels) and
 * deconv_{3,2,1}_0 (:115-121).  big: bf16 [B,Db,Hb,Wb,Cb], Cb in {8,16,32}, Wb even; small: bf16 [B,Ds,Hs,Ws,Cs], Cs in
 * {16,32,64} or a multiple of 16 in (64,128], Ws <= 255; small_strides4_host: NULL (dense) or the (batch, plane, line, voxel)
 * strides of small in elements (HOST int64; a box inside a larger channel-last allocation); gw: fp32 [27,Cb,Cs], zeroed by the
 * call; pad in {1,2}. */
int mvsb200_conv3d_s2_wgrad_lines(const void* big, const void* small, float* gw, int B, int Db, int Hb, int Wb, int Cb,
                                  int Ds, int Hs, int Ws, int Cs, int pad_d, int pad_h, int pad_w,
                                  const int64_t* small_strides4_host, void* stream);

/* Stride-2 TRANSPOSED convolution forward in ONE launch (ConvTranspose3d k=3, scripts/model.py:229-234, used at :115-121):
 *   out[2J + par] = sum over the taps k with (par + pad - k) even of W[k] . in[J + (par + pad - k)/2] per axis.
 * All 8 output-parity classes are accumulated side by side in TMEM and written interleaved, so every line of the canvas is
 * written once, contiguously.  x: [B, Di, Hi, Wi, Cin] bf16 (the central box); w_packed: [28, n_rows, Cin] bf16 (tap 27 = zeros) with tap k
 * = (kd,kh,kw) of the transposed-conv weight, rows = output channels (n_rows 16 or 32); y: voxel row of output (b,z,y,x) at
 * y + b*ys[0] + z*ys[1] + y*ys[2] + x*ys[3] elements (HOST int64), written for z < Do, y < Ho, x < Wo; pad in {1,2}. */
int mvsb200_deconv3d_s2_fwd(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                            int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                            const int64_t* y_strides4_host, void* stream);

/* mvsb200_deconv3d_s2_fwd that also writes, per CTA, the sums of the stored values and of their squares per output channel over
 * the written canvas: stats [n_blocks][2][cout] fp32 (NULL: none), n_blocks returned through n_blocks_host (<= the SM count: size
 * the buffer for that).  With mvsb200_bn_finalize_affine the BatchNorm that follows the transposed convolution
 * (scripts/model.py:115-121: ReLU(BN(deconv))) needs no statistics pass over the canvas. */
int mvsb200_deconv3d_s2_fwd_stats(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                  int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                  const int64_t* y_strides4_host, float* stats, int* n_blocks_host, void* stream);

/* Stride-2 TRANSPOSED convolution whose input channels come as up to three K CHUNKS of 16 / 32 / 64 channels inside a voxel
 * row of x_cs channels (deconv3d_s2_kc_kernel, csrc/conv3d_s2_bwd.cu): the data gradient of the stacked stride-2 branches
 * conv_{1,2,3}_0 (scripts/model.py:104-110) -- 16 + 32 + 64 gradient channels on the central box -> the 32-channel canvas --
 * replacing aten::convolution_backward's data gradient.  out[2J + par] = sum_k W[k] . x[J + (par + pad - k)/2] as above.
 * x: [B, Di, Hi, Wi, x_cs] bf16 dense; w_packed: chunk after chunk, each [28, n_rows, kc_n[c]] bf16 with a 28th all-zero tap (rows = output channels);
 * kc_off / kc_n: HOST int arrays; y as in mvsb200_deconv3d_s2_fwd, cout <= n_rows <= 64; accumulate = 1 adds to y. */
/* Eval-mode form of mvsb200_deconv3d_s2_fwd: the BatchNorm (running statistics) + ReLU that follows the transposed convolution and
 * the skip addition after it (scripts/model.py:117-123, relu(BN(deconv(x))) + enc) in the epilogue, on a WINDOW of the canvas:
 *   y[v] = relu(acc[v] * scale[c] + shift[c]) + add[v][c]      (fp32, one rounding to bf16)
 * for the voxels v of the box window6_host = {lo_d, lo_h, lo_w, n_d, n_h, n_w} (HOST ints) of the Do x Ho x Wo canvas, written in the
 * window's frame: y and add (NULL: no addition; else bf16 rows with y's strides) point at the window's origin voxel.  Only the
 * voxel octets that meet the window are computed.  scale / shift: fp32 [cout] device vectors.  Other arguments as
 * mvsb200_deconv3d_s2_fwd; stored values are bit-identical to that window of relu(acc * scale + shift) (+ add) on the full canvas. */
int mvsb200_deconv3d_s2_fwd_affine(const void* x, const void* w_packed, void* y, int B, int Di, int Hi, int Wi, int Cin,
                                   int Do, int Ho, int Wo, int cout, int n_rows, int pad_d, int pad_h, int pad_w,
                                   const int* window6_host, const int64_t* y_strides4_host, const float* scale, const float* shift,
                                   const void* add, void* stream);

int mvsb200_deconv3d_s2_kc_fwd(const void* x, int x_cs, const void* w_packed, const int* kc_off_host, const int* kc_n_host, int n_kc,
                               void* y, int B, int Di, int Hi, int Wi, int Do, int Ho, int Wo, int cout, int n_rows,
                               int pad_d, int pad_h, int pad_w, const int64_t* y_strides4_host, int accumulate, void* stream);

/* Stride-2 convolution forward on tcgen05 (parity-deinterleaved sub-lattice slabs through TMA): the three stride-2
 * branches conv_{1,2,3}_0 (scripts/model.py:104-110; padding dim/2+1 of scripts/config.py:20 reduces on the central
 * box to pad 1 or 2) stacked along Cout, and the data gradient of the transposed convolutions.
 *   out(z,y,x) = sum_k W[k] . x(2z - pad_d + kd, 2y - pad_h + kh, 2x - pad_w + kw), zero outside x; pad in {1,2}.
 * x: [B, Dx, Hx, Wx, Cin] bf16; w_packed: [27, n_rows, Cin] bf16 (n_rows % 16 == 0, <= 128); y: [B, Do, Ho, Wo, y_cs] bf16. */
int mvsb200_conv3d_s2_fwd(const void* x, const void* w_packed, void* y, int B, int Dx, int Hx, int Wx, int Cin,
                          int Do, int Ho, int Wo, int cout, int y_cs, int n_rows, int pad_d, int pad_h, int pad_w,
                          void* stream);
/* mvsb200_conv3d_s2_fwd that also leaves sums[2][cout] = per-channel (sum, sum of squares) of its outputs, accumulated in the
 * kernels' epilogues from the fp32 accumulators and combined in fixed order -- the box BatchNorm that follows the stacked
 * branches (scripts/model.py:104-110) needs no pass over them for its statistics.  workspace: (SM count) * 2 * cout floats. */
int mvsb200_conv3d_s2_fwd_stats(const void* x, const void* w_packed, void* y, int B, int Dx, int Hx, int Wx, int Cin, int Do, int Ho,
                                int Wo, int cout, int y_cs, int n_rows, int pad_d, int pad_h, int pad_w, float* workspace,
                                float* sums, void* stream);

/* Weight gradient of the same convolution on tcgen05 (autograd of scripts/model.py:101-113 w.r.t. the filters):
 *   gW[tap][ci][co] = sum_v x(v + tap + off)[ci] * gy(v)[co]
 * x: [B, Di, Hi, Wi, Cin] bf16; gy: [B, Do, Ho, Wo, cout] bf16 (cout in {8,16,32,64}); gw: [27, Cin, cout] fp32,
 * ZEROED BY THIS CALL, then accumulated with fp32 reductions (summation order across CTAs is not fixed). */
int mvsb200_conv3d_s1_wgrad(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Cin,
                            int Do, int Ho, int Wo, int cout, int off_d, int off_h, int off_w, void* stream);

/* Per-channel algebra of the box BatchNorm of the stride-2 branches (scripts/model.py:104-110 + BN + ReLU, evaluated on the
 * central box: the canvas outside it is zero and counts in the statistics), one launch each instead of ~12 / ~20 [C]-sized torch
 * launches: forward = mean, biased variance, scale, shift (fp64 inside), the running-statistics update of torch.nn.BatchNorm and
 * stat64 = [mean, 1/sqrt(var + eps)] in fp64 for the backward; backward = (a, b2) = (dL/d sum S, 2 dL/d sum S^2) for
 * mvsb200_box_bn_relu_bwd_apply plus the gradients of gamma and beta, from the reduced (gscale, gshift) and optional external
 * gradients of scale / shift (NULL = none).  add1 / add2 (fp64, NULL = none): what the tensor contributes to the two sums outside
 * the box it was summed over (conv_{1,2,3}_1: closed-form border classes, mvs_b200/regulariser.py). */
/* Closed-form statistics of a stride-1, padding-1 convolution OUTSIDE its computed box when its input is the per-channel constant
 * bg there (second-stage branches conv_{1,2,3}_1, scripts/model.py:105-110): val[co][27 border classes] = sum over the taps that stay
 * on the canvas of sum_ci W[co][ci][tap] bg[ci]; A1 = sum_cls cnt val, A2 = sum_cls cnt val^2 (fp64).  W: fp32 [Cout][Cin][27],
 * cnt27: voxels per class (fp32).  Backward: gW [Cout][Cin][27], gbg [Cin] from (gA1, gA2) (either may be NULL);
 * dt_workspace: Cout * 27 floats. */
int mvsb200_outside_sums_fwd(const float* W, const float* bg, const float* cnt27, int Cout, int Cin, double* val, double* A1,
                             double* A2, void* stream);
int mvsb200_outside_sums_bwd(const float* W, const float* bg, const float* cnt27, const double* val, const double* gA1,
                             const double* gA2, int Cout, int Cin, float* dt_workspace, float* gW, float* gbg, void* stream);
int mvsb200_box_bn_algebra_fwd(const float* s1, const float* s2, const double* add1, const double* add2, int C, double n_full,
                               const float* gamma, const float* beta,
                               double eps, double momentum, float* running_mean, float* running_var,
                               int64_t* num_batches_tracked, float* scale, float* shift, float* mean, float* var,
                               double* stat64, void* stream);
int mvsb200_box_bn_algebra_bwd(const float* gscale, const float* gshift, const float* gscale_ext, const float* gshift_ext,
                               const double* stat64, const float* gamma, int C, double n_full, float* a, float* b2,
                               float* g_gamma, float* g_beta, void* stream);

/* ---- K3c: the output convolution 8 -> 1 channels (k = 3, stride 1, padding 1) -----------------------
 * Replaces conv_out = Conv3d(8, 1, 3, padding=1, bias=False) (scripts/model.py:91, used at :123) and its two
 * gradients.  z: [B, D, h, w, 8] bf16 (the sum y1 + y0, channels_last_3d); w27x8: [27, 8] fp32, tap-major
 * (kd, kh, kw) then input channel; logits / glogits: [B, D, h, w] fp32; gz: [B, D, h, w, 8] bf16;
 * gw27x8: [27, 8] fp32 (deterministic reduction); workspace: mvsb200_conv_out_workspace_floats() floats. */
int64_t mvsb200_conv_out_workspace_floats(void);
int mvsb200_conv_out_fwd(const void* z, const float* w27x8, float* logits, int B, int D, int h, int w, void* stream);
int mvsb200_conv_out_dgrad(const float* glogits, const float* w27x8, void* gz, int B, int D, int h, int w, void* stream);
int mvsb200_conv_out_wgrad(const void* z, const float* glogits, float* workspace, float* gw27x8, int B, int D, int h,
                           int w, void* stream);

/* ---- K3b: train-mode BatchNorm3d (+ReLU) on channel-last volumes -----------------------------------
 * Replaces the BatchNorm3d + ReLU pairs of CostVolumeReg.forward (scripts/model.py:101-121; layer
 * factory :241-247) in train mode (batch statistics over B, D, h, w; scripts/train.py:61, test.py:61).
 * x, y, gy, dx: [M, C] rows of C contiguous channels (a [B,C,D,h,w] volume in channels_last_3d
 * strides, M = B*D*h*w), dtype MVSB200_F32 or MVSB200_BF16; C in {8,16,32,64}.  Per-channel vectors
 * are fp32 [C].  `workspace` is caller-owned scratch of mvsb200_bn_workspace_floats() floats.
 *   bn_stats     mean[c], biased variance[c] of x (deterministic two-stage reduction, fp64 finalize)
 *   bn_relu_fwd  y = x*scale + shift, then max(.,0) if relu        (scale = gamma/sqrt(var+eps))
 *   bn_relu_bwd  dbeta = sum g, dgamma = sum g*xhat, dx = gamma*invstd*(g - dbeta/M - xhat*dgamma/M)
 *                with g = gy * [x*scale+shift > 0] (or gy when !relu), xhat = (x-mean)*invstd */
int64_t mvsb200_bn_workspace_floats(void);
int mvsb200_bn_stats(const void* x, int dtype, int64_t M, int C, float* workspace, float* mean, float* var,
                     void* stream);
int mvsb200_bn_relu_fwd(const void* x, int dtype, const float* scale, const float* shift, void* y, int relu,
                        int64_t M, int C, void* stream);
int mvsb200_bn_relu_bwd(const void* x, int x_dtype, const void* gy, int g_dtype, const float* scale,
                        const float* shift, const float* mean, const float* invstd, const float* gamma,
                        float* workspace, float* dbeta, float* dgamma, void* dx, int relu, int64_t M, int C,
                        void* stream);

/* bn_stats (geo12_host = NULL) or bn_stats_geo followed by the WHOLE per-channel algebra of a train-mode BatchNorm
 * (torch.nn.BatchNorm3d / 2d as built by scripts/model.py:236-247) in one finalize launch: mean, biased variance,
 * invstd = 1/sqrt(var + eps), scale = gamma*invstd, shift = beta - mean*scale and, when running_mean / running_var are given,
 * running = (1 - momentum)*running + momentum*(mean | var*M/(M-1)), *num_batches_tracked += 1 (may be NULL). */
int mvsb200_bn_stats_affine(const void* x, int dtype, int64_t M, int C, float* workspace, const int* geo12_host,
                            const float* gamma, const float* beta, double eps, double momentum, float* running_mean,
                            float* running_var, int64_t* num_batches_tracked, float* mean, float* var, float* invstd,
                            float* scale, float* shift, void* stream);

/* The finalize launch of mvsb200_bn_stats_affine alone, on per-CTA partial sums [n_blocks][2][C] a producer kernel already wrote
 * (mvsb200_deconv3d_s2_fwd_stats); M = the number of voxels per channel the sums run over. */
int mvsb200_bn_finalize_affine(const float* partials, int n_blocks, int64_t M, int C, const float* gamma, const float* beta,
                               double eps, double momentum, float* running_mean, float* running_var,
                               int64_t* num_batches_tracked, float* mean, float* var, float* invstd, float* scale,
                               float* shift, void* stream);

/* Geometry-aware variants.  The canvas [D,h,w] (what the statistics are taken over; M = B*D*h*w) sits at the origin
 * of a possibly larger allocation [Da,ha,wa] (the library's stride-2 transposed convolution returns one extra
 * plane/line/column that the reference crops away, scripts/config.py:21 OUTPAD), and y / gy live only on a box of the
 * canvas (the normalised result is read only on the central box, regulariser.py).
 * geo12 (HOST ints) = {Da, ha, wa, D, h, w, d0, h0, w0, dc, hc, wc};
 * x, dx: [B, Da, ha, wa, C] (dx is 0 outside the canvas); y, gy: [B, dc, hc, wc, C]. */
int mvsb200_bn_stats_geo(const void* x, int dtype, int64_t M, int C, float* workspace, float* mean, float* var,
                         const int* geo12_host, void* stream);
int mvsb200_bn_relu_fwd_crop(const void* x, int dtype, const float* scale, const float* shift, void* y, int relu,
                             int64_t M, int C, const int* geo12_host, void* stream);
/* y = round(max(x*scale + shift, 0)) + add: BatchNorm apply + ReLU + skip addition in one pass (SURVEY §8b `bn_relu_add_apply`;
 * scripts/model.py:117-123).  geo12 == NULL: x, add, y are [M, C] rows; otherwise y and add live on the crop box of x's canvas
 * (geometry as mvsb200_bn_relu_fwd_crop).  The normalised value is rounded to the storage type before the addition: the result
 * equals a separate addition of the stored tensor bit for bit. */
int mvsb200_bn_relu_add_apply(const void* x, int dtype, const float* scale, const float* shift, const void* add, void* y, int relu,
                              int64_t M, int C, const int* geo12, void* stream);
int mvsb200_bn_relu_bwd_crop(const void* x, int x_dtype, const void* gy, int g_dtype, const float* scale,
                             const float* shift, const float* mean, const float* invstd, const float* gamma,
                             float* workspace, float* dbeta, float* dgamma, void* dx, int relu, int64_t M, int C,
                             const int* geo12_host, void* stream);

/* ---- K3d: per-channel sums and affine+ReLU over boxes of channel-last volumes -------------------------
 * The BatchNorm3d + ReLU pairs of the stride-2 branches (scripts/model.py:104-113) evaluated on the central box
 * where those layers carry data (padding dim/2+1, scripts/config.py:20); the constant remainder of the canvas enters
 * the statistics analytically on the host (mvs_b200/regulariser.py).
 * x: a [B, C, D, h, w] view with unit channel stride; strides4 (HOST int64, elements) = {b, d, h, w}; dims4 (HOST)
 * = {B, D, h, w}; C in {8,16,32,64}; dtype f32/bf16.  workspace: mvsb200_affine_workspace_floats() floats.
 *   channel_sums        s1[c] = sum x, s2[c] = sum x^2 (deterministic);  _bwd: gx = g1[c] + 2 x g2[c]  (dense)
 *   affine_relu_geo     geo13 (HOST) = {B, Id, Ih, Iw, in_origin[3], out_origin[3], out_dims[3]} in one frame:
 *                       y(p) = max(xv(p) scale[c] + shift[c], 0) on the output box, xv = x inside the input box, 0 outside.
 *                       y, gy: dense [B, od, oh, ow, C]; gx: dense over the input box; gscale/gshift: [C]. */
int64_t mvsb200_affine_workspace_floats(void);
int mvsb200_channel_sums(const void* x, int dtype, const int64_t* strides4_host, const int* dims4_host, int C,
                         float* workspace, float* s1, float* s2, void* stream);
int mvsb200_channel_sums_bwd(const void* x, int dtype, const int64_t* strides4_host, const int* dims4_host, int C,
                             const float* g1, const float* g2, void* gx, void* stream);
int mvsb200_affine_relu_geo_fwd(const void* x, int dtype, const int64_t* strides4_host, const int* geo13_host, int C,
                                const float* scale, const float* shift, void* y, int relu, void* stream);
int mvsb200_affine_relu_geo_bwd(const void* x, int x_dtype, const int64_t* strides4_host, const int* geo13_host, int C,
                                const float* scale, const float* shift, const void* gy, int g_dtype, float* workspace,
                                float* gscale, float* gshift, void* gx, int relu, void* stream);

/* Train-mode BatchNorm3d + ReLU of a stride-2 branch on its central box (scripts/model.py:104-110 with the padding of
 * scripts/config.py:20), backward in two halves around the per-channel algebra of the statistics:
 *   reduce  gshift[c] = sum g, gscale[c] = sum g * xv,  g = gy * [xv*scale+shift > 0]   (over the output box)
 *   apply   gx = g * scale + a + b2 * xv   over the input box, with a = dL/d(sum x), b2 = 2 dL/d(sum x^2): ONE pass instead of
 *           an affine data gradient, a statistics gradient and their sum; gx (x's dtype) is written through out_strides4_host
 *           (elements) so that it can land inside the padded, channel-stacked buffer the strided convolution's backward reads. */
int mvsb200_box_bn_relu_bwd_reduce(const void* x, int x_dtype, const int64_t* strides4_host, const int* geo13_host, int C,
                                   const float* scale, const float* shift, const void* gy, int g_dtype, float* workspace,
                                   float* gscale, float* gshift, int relu, void* stream);
int mvsb200_box_bn_relu_bwd_apply(const void* x, int x_dtype, const int64_t* strides4_host, const int* geo13_host, int C,
                                  const float* scale, const float* shift, const float* a, const float* b2, const void* gy,
                                  int g_dtype, void* gx, const int64_t* out_strides4_host, int relu, void* stream);

/* ---- f3: the training loss (SURVEY §8 row f3; scripts/loss.py:4-41), fused ------------------------------------------
 * mask = (gt != 0), n_valid[b] = sum mask;  l0[b] = sum mask |gt - initial| / n_valid[b], l1[b] likewise for `refined`;
 * out3 = (loss = sum_b l0 + l1, initial_acc = mean_b l0, refined_acc = mean_b l1): one launch (32 CTAs per sample, the last to
 * finish combines them, fixed order).  Backward: one elementwise launch, g3 = device floats (dL/d loss, dL/d initial_acc,
 * dL/d refined_acc).  gt / initial / refined: fp32 [B, n] dense; workspace: mvsb200_masked_l1_workspace_floats(B) floats, ZEROED
 * once by the caller (its last word is the ticket counter, reset by every launch); it carries (n_valid, l0, l1) to the backward. */
int64_t mvsb200_masked_l1_workspace_floats(int B);
int mvsb200_masked_l1_fwd(const float* gt, const float* initial, const float* refined, int B, int n, float* workspace,
                          float* out3, void* stream);
int mvsb200_masked_l1_bwd(const float* gt, const float* initial, const float* refined, const float* workspace,
                          const float* g3, int B, int n, float* g_initial, float* g_refined, void* stream);

/* ---- f2: the glue either side of the depth-refinement network (SURVEY §8 row f2; scripts/model.py:190-205) -------------
 * refine_input_fwd:  norm = (initial - d_min[b]) / span[b] (fp32 [B, h*w]) and the network's input as bf16 channel-last rows
 *                    [B, h, w, cp] (cp = 8 or 16): channel 0 = norm, 1..3 = the reference image (view b * n_views of `images`, fp32
 *                    [N, 3, H, W] with the given element strides) resized to h x w as torch's bilinear interpolate (align_corners =
 *                    False) does, the remaining channels zero (what the K = 16 tensor-core convolution reads).
 * refine_input_bwd:  g_initial = (g_rows[., 0] + g_norm) / span[b]; either gradient may be NULL.
 * refine_output_fwd: refined = (res_rows[., 0] + norm) * span[b] + d_min[b]   (model.py:150-151 and :203).
 * refine_output_bwd: g_rows [B*n, cr] bf16 (channel 0 = g * span[b], others zero; cr = 8 or 16) and g_norm = g * span[b]. */
int mvsb200_refine_input_fwd(const float* initial, const float* images, const int64_t* image_strides4_host, int n_views, int H, int W,
                             const float* d_min, const float* span, int B, int h, int w, int cp, void* rows, float* norm,
                             void* stream);
int mvsb200_refine_input_bwd(const void* g_rows, int cp, const float* g_norm, const float* span, int B, int n, float* g_initial,
                             void* stream);
int mvsb200_refine_output_fwd(const void* res_rows, int cr, const float* norm, const float* d_min, const float* span, int B, int n,
                              float* refined, void* stream);
int mvsb200_refine_output_bwd(const float* g_refined, const float* span, int B, int n, int cr, void* g_rows, float* g_norm,
                              void* stream);

/* ---- f1: the 2D feature encoder on the path's kernels (SURVEY §8 row f1; scripts/model.py:22-65) ------------------------
 * Maps travel as channel-last bf16 rows, stacked as the planes of ONE volume [1, C, N, H, W]: a 3x3 convolution is the middle
 * depth slice of a 3x3x3 one (mvsb200_pack_filter with the kd = 0 / 2 slots empty, mvsb200_conv3d_s1_fwd_kdn), its weight gradient
 * mvsb200_conv3d_s1_wgrad_ex with kd_mask = 2; a 5x5 stride-2 convolution is a 3x3 one on the space-to-depth form of its input.
 * image_to_rows8:  fp32 [N, 3, H, W] (element strides given) -> bf16 rows [N, H, W, 8], channels 3..7 zero.
 * s2d_rows_bf16:   [N, 2h, 2w, C] -> [N, h, w, 4C] (channel (py*2 + px)*C + c), inverse != 0: the other way.  C % 8 == 0.
 * conv3d_s1_wgrad_ex: mvsb200_conv3d_s1_wgrad with a depth-tap mask (bit kd: compute that tap's gradient, the others stay zero)
 *                  and Cin = 8 (8-channel rows on the K = 16 kernel; gw is then [27][16][cout], rows 8..15 zero).
 * conv2d_rows_fwd:  3x3 / padding-1 convolution of N stacked maps, rows [N, H, W, Cin] -> [N, H, W, y_cs]: conv3d_s1_kdn_kernel in its
 *                  planar mode (MMAs of N = cout on the middle depth slice of the kdn filter operand [9][3][n_rows][Cin], one slab
 *                  per map, no halo planes); with the flipped, transposed filter it is the data gradient. */
/* BatchNorm apply + ReLU written straight in the space-to-depth form (x rows [N, H, W, C] bf16 -> y rows [N, H/2, W/2, 4C], M = N*H*W),
 * and the BatchNorm backward that reads its incoming gradient gy from that form (dx in x's form): the permutation in front of a 5x5
 * stride-2 layer costs no pass of its own.  Arguments as mvsb200_bn_relu_fwd / mvsb200_bn_relu_bwd (bf16 x, y, gy, dx). */
int mvsb200_bn_relu_fwd_s2d(const void* x, int dtype, const float* scale, const float* shift, void* y, int relu, int64_t M, int C,
                            int H, int W, void* stream);
int mvsb200_bn_relu_bwd_s2d(const void* x, const void* gy, const float* scale, const float* shift, const float* mean,
                            const float* invstd, const float* gamma, float* workspace, float* dbeta, float* dgamma, void* dx,
                            int relu, int64_t M, int C, int H, int W, void* stream);
int mvsb200_conv2d_rows_fwd(const void* x, const void* w_packed, void* y, int N, int H, int W, int Cin, int cout, int y_cs, int n_rows,
                            void* stream);
int mvsb200_image_to_rows8(const float* images, const int64_t* strides4_host, int N, int H, int W, void* rows, void* stream);
int mvsb200_s2d_rows_bf16(const void* src, void* dst, int N, int h, int w, int C, int inverse, void* stream);
int mvsb200_conv3d_s1_wgrad_ex(const void* x, const void* gy, float* gw, int B, int Di, int Hi, int Wi, int Cin, int Do, int Ho,
                               int Wo, int cout, int off_d, int off_h, int off_w, unsigned kd_mask, void* stream);

/* ---- K7: multi-view consistency filter and point-cloud fusion (MVSNet §4.2) -----------------------------------------------------
 * N depth maps [N, h, w] of one scene, their confidences, and a camera table cams [N, MVSB200_FUSION_CAM_FLOATS] fp32 per view:
 *   [0:12] P = K [R | T] (3x4, row-major)  [12:21] R^T K^-1  [21:24] C = -R^T T  [24:27] n, the depth normal  [27:32] unused.
 * Depth d at pixel (x, y) is the point X = C + d / (n^T r) r with r = R^T K^-1 (x, y, 1); the depth of X in view j is n_j^T (X - C_j).
 * sources [N, S] int32 (S <= 16, -1 = padding).  A pixel is valid when conf >= conf_min and d is finite and > 0; a source s is
 * consistent when X projects into s with z > 0 inside [0, w-1] x [0, h-1], the four bilinear taps of d_s there are finite and > 0,
 * and the point X_s (the sampled depth unprojected in s) projects back to p' with |p' - p| < reproj_px and
 * |n_ref^T (X_s - C_ref) - d| / d < rel_depth.  mask = valid && count >= min_views, fused = (d + sum of reprojected depths) /
 * (1 + count).  block_counts [N * ceil(h w / MVSB200_FUSION_BLOCK_PIXELS)]: the masked pixels of each block (view-major). */
#define MVSB200_FUSION_CAM_FLOATS 32
#define MVSB200_FUSION_BLOCK_PIXELS 128
#define MVSB200_FUSION_MAX_SOURCES 16
int mvsb200_fusion_check(const float* depth, const float* conf, const float* cams, const int32_t* sources, int N, int S,
                         int h, int w, float conf_min, float reproj_px, float rel_depth, int min_views,
                         uint8_t* mask, int32_t* count, float* fused, int32_t* block_counts, void* stream);

/* compaction: offsets [N * blocks] int64, the exclusive scan of block_counts.  Writes xyz [M, 3] (the fused depth unprojected at the
 * reference pixel) and rgb [M, 3] (colours [N, 3, h, w] at that pixel) in view-major, row-major order; deterministic, no atomics. */
int mvsb200_fusion_emit(const uint8_t* mask, const float* fused, const float* colours, const float* cams, const int64_t* offsets,
                        int N, int h, int w, float* xyz, float* rgb, void* stream);

/* images [N, 3, H, W] fp32 contiguous -> out [N, 3, h, w]: torch's bilinear resize with align_corners = False (as refine_input) */
int mvsb200_resize_rgb(const float* images, int N, int H, int W, int h, int w, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MVS_B200_H_ */
