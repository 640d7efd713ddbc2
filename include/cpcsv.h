/*
 * cpcsv.h -- C ABI of libcpcsv.so, the sm_100a kernels behind the CP-CSV drop-in modules.
 *
 * The reference (basiclab/CPCStoryVisualization-Pytorch) has no FFI of its own: its hot path
 * is PyTorch calls inside model.py / layers.py.  Each entry point below replaces the library
 * kernels PyTorch dispatches to for one reference call site (cited per function, paths are
 * into the reference tree).  INTEGRATION.md shows the ctypes binding model.py uses.
 *
 * Conventions (SURVEY.md section 8b)
 *  - plain pointers and sizes only; the caller owns every buffer; nothing is retained.
 *  - enqueue-only on `stream`; no synchronisation, no device allocation; graph-capturable.
 *  - return 0 on success, <0 argument error (nothing enqueued), >0 cudaError_t.
 *    cpcsv_last_error_string() describes the last failure on the calling thread.
 *  - activations are NHWC; "pix" = flattened (n,h,w); 16-bit operand tensors are bf16
 *    unless dtype says fp16; statistics, accumulators and gradients are fp32.
 */
#ifndef CPCSV_H_
#define CPCSV_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* cpcsv_stream_t; /* cudaStream_t */

int cpcsv_version(void);
const char* cpcsv_last_error_string(void);
/* number of kernels this library has enqueued from the calling process so far */
int64_t cpcsv_launch_count(void);

/* ------------------------------------------------------------------ tcgen05 implicit GEMM
 * One kernel family serves every convolution / transposed convolution / weight-gradient /
 * large Linear on the path:
 *   model.py:16-34   conv3x3, upBlock (nearest x2 + conv3x3, executed as 4 sub-pixel 2x2 convs)
 *   model.py:260-263,285-288  fc / fc_seg Linear
 *   model.py:278-279 seg_c / seg_c1
 *   model.py:498-514,540-556,582-598  D encoders (conv 4x4 stride 2)
 *   model.py:75-80   D_GET_LOGITS conv3x3 over [features | tiled condition]
 * and their autograd backward passes (dgrad = same kernel with transposed weights,
 * wgrad = mode 1).
 *
 * A 16-bit operand is described as a 5-D strided view (c, w, p, h, n): c contiguous.  For a
 * plain NHWC tensor p has extent 1; for stride-2 access the tensor is viewed as
 * (2C, W/2, 2, H/2, N) so that a "tap" selects the row/column parity through (p, c-offset).
 * TMA zero-fills out-of-range coordinates, which implements the convolution padding.
 */
typedef struct {
  const void* ptr;
  int64_t dims[5];    /* elements: c, w, p, h, n */
  int64_t strides[5]; /* bytes; strides[0] is ignored (elements are contiguous in c) */
} cpcsv_view5_t;

typedef struct {
  int32_t a[4]; /* added to the A-operand TMA coordinate: (c, w, p, h) */
  int32_t b[4]; /* mode 0: b[0] = first weight row of this tap; mode 1: (c, w, p, h) of B */
  int64_t out_off; /* element offset into `out`: mode 0 read from the first tap of a group
                      (sub-pixel phase offset); mode 1 per tap (one matrix per tap) */
} cpcsv_tap_t;

#define CPCSV_MAX_TAPS 16

typedef struct {
  int32_t mode;   /* 0: D[pix, cout] = sum_taps A_tap[pix, k] * B_tap[cout, k]   (K-major operands)
                     1: D_tap[ca, cb] = sum_pix A_tap[pix, ca] * B_tap[pix, cb]  (MN-major operands) */
  int32_t dtype;  /* 0 = fp16, 1 = bf16 */
  int32_t planes; /* 1: single pass; 2: hi/lo split operands, 3 MMAs (hi*hi + lo*hi + hi*lo) */
  int32_t N, H, W;                /* pixel grid the tiles walk over */
  int32_t tile_n, tile_h, tile_w; /* pixel box: product 128 (mode 0) or 64 (mode 1) */
  int32_t groups;                 /* mode 0: sub-pixel phases; mode 1: number of taps */
  int32_t taps_per_group;         /* mode 0 only (mode 1: 1) */
  int32_t k_blocks;               /* mode 0: reduction channels / 64 */
  int32_t m_valid;                /* mode 1: valid rows (A channels) */
  int32_t n_valid;                /* valid output columns (<= n_tiles * block_n) */
  int32_t block_n;                /* 16..256, multiple of 16 */
  int32_t n_tiles;
  int32_t splits;                 /* split-K factor (>1 forces atomic accumulation) */
  int32_t accumulate;             /* 1: add into `out` instead of overwriting */
  int32_t cta_pair;               /* 1 = run as cta_group::2 pairs: two CTAs of a cluster (two 128-row M tiles)
                                     share every B tile, each loading half of it -- half the B traffic per SM.
                                     mode 0: block_n >= 32 in steps of 16; mode 1: block_n 128 or 256 (whole
                                     64-channel atoms per CTA).  Pays off on long jobs, costs a few microseconds
                                     of cluster launch on short ones */
  int64_t out_stride_n, out_stride_h, out_stride_w; /* mode 0: elements per pixel step */
  int64_t ldc;                    /* mode 1: row pitch of each output matrix (elements) */
  const float* alpha;             /* optional device scalar multiplied into the result */
  float* out;
  double* stats;                  /* optional (mode 0, splits == 1, accumulate == 0): per-column sum and
                                     sum of squares of the stored values over the valid rows, ADDED into
                                     stats[col] and stats[stats_ld + col] -- the BatchNorm batch statistics
                                     of the conv output (model.py:31-32) without a pass over it */
  int64_t stats_ld;
  cpcsv_view5_t a[2];             /* hi, lo */
  cpcsv_view5_t b[2];             /* hi, lo; mode 0: dims (k, rows, 1, 1, 1) */
  cpcsv_tap_t taps[CPCSV_MAX_TAPS];
} cpcsv_gemm_t;

int cpcsv_conv_gemm(const cpcsv_gemm_t* job, cpcsv_stream_t stream);

/* -------------------------------------------------------- BatchNorm / activation / packing
 * nn.BatchNorm2d / BatchNorm1d in train mode + ReLU / LeakyReLU(0.2) (model.py:32-33,
 * 252-263, 503-513; semantics SURVEY.md Appendix A) on fp32 [rows, C] conv outputs, fused
 * with the split into bf16 hi/lo operand planes for the next tcgen05 GEMM.
 */
/* per-channel sum and sum of squares (fp64), ADDED into stats[0..C) (sum) and stats[C..2C) (sumsq):
 * the caller zeroes `stats` (2C doubles = cpcsv_bn_workspace_doubles) before the first contribution.
 * Contributions may also come from the epilogue of cpcsv_conv_gemm (cpcsv_gemm_t.stats), in which
 * case this pass over the conv output is not needed at all.  Same convention for `sums` of
 * cpcsv_bn_bwd_reduce. */
int64_t cpcsv_bn_workspace_doubles(int64_t rows, int32_t C);
int cpcsv_bn_stats(const float* x, int64_t rows, int32_t C, int64_t ldx, double* stats,
                   cpcsv_stream_t stream);
/* mean/invstd, running-stat update (momentum 0.1, unbiased var), scale/shift.
 * chan_map (optional) maps local channel j -> index into gamma/beta/running_* (fc layers
 * run in a permuted channel order).  gamma==NULL: identity affine (no BN).  */
int cpcsv_bn_finalize(const double* stats, int64_t rows, int32_t C, const float* gamma,
                      const float* beta, float* running_mean, float* running_var,
                      const int32_t* chan_map, int32_t C_valid, float eps, float momentum,
                      float* mean, float* invstd, float* scale, float* shift,
                      cpcsv_stream_t stream);
/* y = act(x*scale + shift) [* (1 + mod)]; writes any of: fp32 y, 16-bit hi, 16-bit lo.
 * act: 0 none, 1 ReLU, 2 LeakyReLU(0.2).  scale==NULL: identity.  */
int cpcsv_bn_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx, const float* scale,
                      const float* shift, int32_t act, const float* mod, int64_t ldmod,
                      float* y, int64_t ldy, void* hi, void* lo, int64_t ldp, int32_t dtype,
                      cpcsv_stream_t stream);
/* backward of the above.  dy is the gradient w.r.t. the (modulated) activation.
 *   a   = act(x*scale+shift);  dmod = dy * a;  da = dy * (1 + mod);  g = da * act'(.)
 * pass 1 (reduce): sums[0..C) += sum g, sums[C..2C) += sum g * xhat  (fp64; caller-zeroed)
 * pass 2 (apply):  dx = scale_g * invstd * (g - mean(g) - xhat * mean(g*xhat))      */
int cpcsv_bn_bwd_reduce(const float* x, const float* dy, int64_t rows, int32_t C, int64_t ldx,
                        int64_t lddy, const float* scale, const float* shift, const float* mean,
                        const float* invstd, int32_t act, const float* mod, int64_t ldmod,
                        double* sums, cpcsv_stream_t stream);
int cpcsv_bn_bwd_apply(const float* x, const float* dy, int64_t rows, int32_t C, int64_t ldx,
                       int64_t lddy, const float* scale, const float* shift, const float* mean,
                       const float* invstd, const float* gamma, const int32_t* chan_map,
                       int32_t C_valid, int32_t act, const float* mod, int64_t ldmod,
                       const double* sums, int32_t has_bn, float* dx, int64_t lddx, void* dx16,
                       int64_t ld16, float* dmod, int64_t lddmod, void* dmod16, int64_t lddmod16,
                       float* dgamma, float* dbeta, cpcsv_stream_t stream);

/* bn_finalize + bn_act_pack in ONE launch: every block derives scale / shift of its channels from
 * the fp64 sums in `stats` (batch statistics over `rows` rows); vec = [mean | invstd | scale | shift]
 * (4*C floats, for the backward pass) and the running statistics are written once. */
int cpcsv_bn_norm_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx, const double* stats,
                           const float* gamma, const float* beta, float* running_mean,
                           float* running_var, const int32_t* chan_map, int32_t C_valid, float eps,
                           float momentum, float* vec, int32_t act, const float* mod, int64_t ldmod,
                           float* y, int64_t ldy, void* hi, void* lo, int64_t ldp, int32_t dtype,
                           cpcsv_stream_t stream);

/* end of an R(2+1)D-18 BasicBlock in eval mode (torchvision.models.video.resnet.BasicBlock, which the
 * reference's fid/residual2p1.py builds and fid/vfid_score.py runs for the story-level FID):
 *   y = act(x*scale + shift + (r*rscale + rshift))
 * x is the fp32 output of the block's last conv, r the shortcut [rows, C] (pitch ldr): the block input
 * (rscale == rshift == NULL, identity shortcut) or the output of its (1,1,1) stride-2 projection conv
 * (rscale / rshift: that branch's eval-mode BatchNorm).  scale / shift: the block's last BatchNorm.
 * Writes any of fp32 y (the next block's identity shortcut), 16-bit hi, 16-bit lo; rows / pitches /
 * channel padding as cpcsv_bn_act_pack (padding channels have zero scale, shift and residual). */
int cpcsv_bn_add_act_pack(const float* x, int64_t rows, int32_t C, int64_t ldx, const float* scale,
                          const float* shift, const float* r, int64_t ldr, const float* rscale,
                          const float* rshift, int32_t act, float* y, int64_t ldy, void* hi, void* lo,
                          int64_t ldp, int32_t dtype, cpcsv_stream_t stream);

/* ------------------------------------------------------------------- frame FID (InceptionV3) */
/* Stem input of the FID InceptionV3 (cpcsv_b200/frame_fid.py): the fp32 NCHW 3-channel frames x [N, 3, H, W]
 * (element strides sn, sc, sh, sw, any size) resized bilinearly to S x S (align_corners=False, no antialias,
 * PyTorch's source-index rule), mapped by v = a * sample + b, and written as the im2col rows of the 3x3 stride-2
 * pad-0 Conv2d_1a_3x3: row (n, oh, ow) of OH = (S - 3) / 2 + 1, column (ky*3 + kx)*3 + c (< 27; columns up to ldp
 * are zero), as 16-bit hi / lo (lo optional) planes with row pitch ldp (a multiple of 8, 16-B aligned planes).
 * The S x S image is never materialised. */
int cpcsv_resize_im2col(const float* x, int32_t N, int32_t H, int32_t W, int64_t sn, int64_t sc, int64_t sh,
                        int64_t sw, int32_t S, float a, float b, void* hi, void* lo, int32_t ldp, int32_t dtype,
                        cpcsv_stream_t stream);
/* 3x3 pooling of a pitched fp32 NHWC input x [N, H, W, C] (pixel pitches sn, sh, sw in elements, channels
 * contiguous, C % 4 == 0): mode 0 max, mode 1 average over the taps inside the input (count_include_pad=False);
 * stride 1 pad 1 (output H x W) or stride 2 pad 0 (output (H - 3) / 2 + 1).  Writes fp32 y (a channel slice of
 * a wider buffer: pitches ysn, ysh, ysw) and / or 16-bit hi / lo planes (pitches psn, psh, psw); all pitches
 * multiples of 4 elements, x / y 16-B and the planes 8-B aligned. */
int cpcsv_pool3x3(const float* x, int32_t N, int32_t H, int32_t W, int32_t C, int64_t sn, int64_t sh, int64_t sw,
                  int32_t mode, int32_t stride, float* y, int64_t ysn, int64_t ysh, int64_t ysw, void* hi, void* lo,
                  int64_t psn, int64_t psh, int64_t psw, int32_t dtype, cpcsv_stream_t stream);

/* ------------------------------------------------------------------- frame SSIM */
/* Per-frame SSIM of the reference's evaluation (ssim_score.py / the SSIM loop of trainer.py:175-182, which call
 * pytorch_ssim.ssim(x, y, size_average=False)): x, y fp32 with logical layout [B, T, C, H, W] and element strides
 * (xsb, xst, xsc, xsh, xsw) / (ysb, ...) -- stories [B, C, T, H, W] without a copy, plain frames as T = 1 -- both
 * mapped by v = a * v + b on load.  out[b * T + t] (fp64) = the mean over C x H x W of the SSIM map of frame (b, t):
 * 11-tap Gaussian window (sigma 1.5, sum 1) per channel, zero padding 5 (border windows see zeros, no
 * renormalisation), sigma^2 = E[v^2] - mu^2, sigma_xy = E[xy] - mu_x mu_y, C1 = 0.01^2, C2 = 0.03^2,
 * ssim = ((2 mu_x mu_y + C1)(2 sigma_xy + C2)) / ((mu_x^2 + mu_y^2 + C1)(sigma_x^2 + sigma_y^2 + C2)).
 * Moments in fp32, the mean in fp64.  Any C, H, W >= 1.  One CTA per frame, no atomics: a frame's value depends
 * only on its own pixels (not on B, its index or the other frames) and is bit-reproducible. */
int cpcsv_ssim(const float* x, const float* y, int32_t B, int32_t T, int32_t C, int32_t H, int32_t W,
               int64_t xsb, int64_t xst, int64_t xsc, int64_t xsh, int64_t xsw,
               int64_t ysb, int64_t yst, int64_t ysc, int64_t ysh, int64_t ysw,
               float a, float b, double* out, cpcsv_stream_t stream);

/* ------------------------------------------------------------------- layout / pack kernels */
/* generated frames / image sheets for the PNG writers (miscc/utils.py:230-235 images_to_numpy,
 * inference.py:181-197): x [C, H, W] fp32 in [-1, 1] with element strides (sc, sh, sw) ->
 * uint8 [H, W, C] = trunc((clip(x, -1, 1) + 1) / 2 * 255) */
int cpcsv_images_to_u8(const float* x, int32_t C, int32_t H, int32_t W, int64_t sc, int64_t sh,
                       int64_t sw, uint8_t* out, cpcsv_stream_t stream);
/* fp32 strided (n, c, h, w) -> NHWC 16-bit hi/lo planes with channel pitch ldp; channels
 * c >= C are zero-filled up to Cpad.  `bcast` (optional, [n, Cb]) is appended after the C
 * tensor channels and broadcast over (h, w): the concat of D_GET_LOGITS (model.py:88-92). */
int cpcsv_pack_nchw(const float* x, int32_t N, int32_t C, int32_t H, int32_t W, int64_t sn,
                    int64_t sc, int64_t sh, int64_t sw, const float* bcast, int32_t Cb,
                    int64_t ldb, void* hi, void* lo, int32_t Cpad, int32_t dtype,
                    cpcsv_stream_t stream);
/* im2col of a small-channel image for the k x k / stride s / pad p conv it feeds:
 * col[(n, oh, ow), (ky*k+kx)*C + c] (pitch ldp, zero padded).  Serves D layer 0
 * (model.py:499,541,583: 4x4 s2 p1 on 3 or 1 channels).  scale_act: 0 none. */
int cpcsv_im2col_small(const float* x, int32_t N, int32_t C, int32_t H, int32_t W, int64_t sn,
                       int64_t sc, int64_t sh, int64_t sw, int32_t k, int32_t s, int32_t p,
                       void* hi, void* lo, int32_t ldp, int32_t dtype, cpcsv_stream_t stream);
/* First discriminator layer in one launch (model.py:498-500, 540-542, 582-584): Conv2d(C, Co, 4, 2, 1,
 * bias=False) of the strided fp32 image x (C = 1 or 3, H % 4 == 0, W % 64 == 0) with the raw weight
 * w [Co, C, 4, 4], * alpha[0] (1 / sigma of the spectral norm, or NULL), LeakyReLU(slope), written as NHWC
 * 16-bit hi / lo (lo optional) planes with channel pitch ldp <= 128 (channels >= Co zero). */
int cpcsv_enc0_lrelu_fwd(const float* x, int32_t N, int32_t C, int32_t H, int32_t W, int64_t sn, int64_t sc,
                         int64_t sh, int64_t sw, const float* w, int32_t Co, const float* alpha, float slope,
                         void* hi, void* lo, int32_t ldp, int32_t dtype, cpcsv_stream_t stream);
/* LeakyReLU backward from the ACTIVATED values' hi plane (the sign survives the activation):
 * dz[i] (bf16) = dy[i] * (a_hi[i] > 0 ? 1 : slope), count % 8 == 0. */
int cpcsv_lrelu_bwd16(const float* dy, const void* a_hi, int64_t count, float slope, void* dz,
                      cpcsv_stream_t stream);
/* adjoint of im2col_small: dx[n, c, h, w] (contiguous NCHW fp32) = sum over taps of dcol */
int cpcsv_col2im_small(const float* dcol, int64_t ldc, int32_t N, int32_t C, int32_t H, int32_t W,
                       int32_t k, int32_t s, int32_t p, float* dx, cpcsv_stream_t stream);
/* img / img_seg heads as a pixel-major GEMM + gather (model.py:272-274,298-300,401-407): z [N*H*W, ldz]
 * fp32 holds Z[p, tap*Co + co] = sum_c a[p, c] * w[co, c, tap] (cpcsv_conv_gemm, N = 9*Co padded);
 * y[n, co, h, w] = tanh(sum over the 3x3 taps of Z at the shifted pixel), zero outside the image. */
int cpcsv_head_gather_tanh(const float* z, int64_t ldz, int32_t N, int32_t H, int32_t W, int32_t Co,
                           float* y, cpcsv_stream_t stream);
/* backward of the heads: dz = dy * (1 - y^2), emitted directly as the 3x3 im2col of dz in
 * 16-bit: col[pix, tap*C + c] = dz[pix - delta_tap, c] (pitch ldp), which is both the dgrad
 * A operand and the wgrad B operand.  dy strided (n, c, h, w). */
int cpcsv_tanh_bwd_im2col(const float* dy, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                          const float* y, int32_t N, int32_t C, int32_t H, int32_t W, void* col,
                          int32_t ldp, int32_t dtype, cpcsv_stream_t stream);
/* fp32 matrix -> 16-bit hi/lo with optional row / column gather, column padding and
 * transposition; the weight re-layout for the GEMM B operand of the Linear layers.
 * out[r, c] = w[rmap(r) * ld_r + cmap(c) * ld_c] for c < cols_valid, else 0 (a negative map
 * entry also gives 0).  Used for fc / fc_seg (model.py:260-263,285-288), whose output
 * features are re-ordered from (c, y, x) to NHWC (y, x, c) at pack time. */
int cpcsv_pack_matrix(const float* w, int64_t rows_out, int64_t cols_out, int64_t cols_valid,
                      int64_t ld_r, int64_t ld_c, const int32_t* row_map, const int32_t* col_map,
                      void* hi, void* lo, int64_t ldo, int32_t dtype, cpcsv_stream_t stream);
/* dst[row_map[r], c] = src[r, c]  (fp32; undoes the row re-ordering for weight gradients) */
int cpcsv_scatter_rows_f32(const float* src, int64_t ld_src, const int32_t* row_map, float* dst,
                           int64_t ld_dst, int64_t rows, int64_t cols, cpcsv_stream_t stream);
/* conv weight [Cout, Cin, kh, kw] fp32 -> tap-major GEMM operands.
 *  kind 0: plain taps          out[tap][co][ci]        (fprop B)
 *  kind 1: plain taps, transposed  out[tap][ci][co]    (dgrad B)
 *  kind 2: sub-pixel merged 2x2 taps of a 3x3 kernel (SURVEY.md Appendix A)
 *          out[phase(a,b)][tap(i,j)][co][ci]           (upBlock fprop B)
 *  kind 3: sub-pixel merged, transposed out[(a,b,i,j)][ci][co]  (upBlock dgrad B)
 * rows are padded to rows_pad and columns to cols_pad with zeros. */
int cpcsv_pack_conv_weight(const float* w, int32_t Cout, int32_t Cin, int32_t kh, int32_t kw,
                           int32_t kind, int32_t rows_pad, int32_t cols_pad, void* hi, void* lo,
                           int32_t dtype, cpcsv_stream_t stream);
/* inverse maps for weight gradients: GEMM wgrad output dwt[tap][ca][cb] (fp32, pitch ldc,
 * matrices of mat_stride elements) -> dW [Cout, Cin, kh, kw], optionally scaled by *alpha.
 *  kind 0: dwt[tap][co][ci]; kind 1: dwt[tap][ci][co];
 *  kind 2: merged sub-pixel dwt[(a,b,i,j)][co][ci] -> 3x3;  kind 3: same with [ci][co]. */
int cpcsv_unpack_conv_wgrad(const float* dwt, int64_t mat_stride, int64_t ldc, int32_t Cout,
                            int32_t Cin, int32_t kh, int32_t kw, int32_t kind, const float* alpha,
                            float* dw, cpcsv_stream_t stream);

/* cpcsv_unpack_conv_wgrad (kinds 0 / 2) that also adds sum(dW .* w) into *dot (caller-zeroed): the scalar
 * of the spectral-norm backward, without another pass over the gradient */
int cpcsv_unpack_conv_wgrad_dot(const float* dwt, int64_t mat_stride, int64_t ldc, int32_t Cout,
                                int32_t Cin, int32_t kh, int32_t kw, int32_t kind, const float* alpha,
                                float* dw, const float* w, float* dot, cpcsv_stream_t stream);

/* ------------------------------------------------------------- conditioning path (fp32)
 * CA_NET (model.py:37-65), GRUCells (model.py:223-224,313-346), m_net/c_net/image_net/
 * filter_net Linear+BN1d (model.py:250-257,302-308), DynamicFilterLayer1D (layers.py:62-80).
 */
/* Y[M,N] = X[M,K] * W[N,K]^T (+ bias) (+= if accumulate); all fp32 row-major with pitches */
int cpcsv_linear_f32(const float* X, int64_t ldx, const float* W, int64_t ldw, const float* bias,
                     float* Y, int64_t ldy, int32_t M, int32_t N, int32_t K, int32_t accumulate,
                     cpcsv_stream_t stream);
/* Y[M,N] = A[K,M]^T * B[K,N]  (weight gradients dW = dY^T X) */
int cpcsv_linear_tn_f32(const float* A, int64_t lda, const float* B, int64_t ldb, float* Y,
                        int64_t ldy, int32_t M, int32_t N, int32_t K, int32_t accumulate,
                        cpcsv_stream_t stream);
/* Y[M,N] = X[M,K] * W[K,N]  (input gradients dX = dY W) */
int cpcsv_linear_nn_f32(const float* X, int64_t ldx, const float* W, int64_t ldw, float* Y,
                        int64_t ldy, int32_t M, int32_t N, int32_t K, int32_t accumulate,
                        cpcsv_stream_t stream);
/* GRUCell gates: gi = x W_ih^T + b_ih, gh = h W_hh^T + b_hh are given ([B, 3H], order r,z,n);
 * h' = (1-z) n + z h.  Saves r, z, n, (W_hn h + b_hn) for backward in `save` [B, 4H]. */
int cpcsv_gru_gates_fwd(const float* gi, const float* gh, const float* h, int32_t B, int32_t H,
                        float* hnew, float* save, cpcsv_stream_t stream);
int cpcsv_gru_gates_bwd(const float* dhnew, const float* h, const float* save, int32_t B,
                        int32_t H, float* dgi, float* dgh, float* dh, cpcsv_stream_t stream);
/* CA_NET: x = relu(pre); mu = x[:, :C]; logvar = x[:, C:]; code = eps*exp(.5 logvar)+mu */
int cpcsv_ca_fwd(const float* pre, const float* eps, int32_t B, int32_t C, float* mu,
                 float* logvar, float* code, cpcsv_stream_t stream);
int cpcsv_ca_bwd(const float* pre, const float* eps, const float* dmu, const float* dlogvar,
                 const float* dcode, int32_t B, int32_t C, float* dpre, cpcsv_stream_t stream);
/* DynamicFilterLayer1D: out[i, x] = sum_c sum_k img[i, c, x + k - K/2] * filt[i, c, k] */
int cpcsv_dfn1d_fwd(const float* img, const float* filt, int32_t N, int32_t C, int32_t L,
                    int32_t K, float* out, cpcsv_stream_t stream);
int cpcsv_dfn1d_bwd(const float* img, const float* filt, const float* dout, int32_t N, int32_t C,
                    int32_t L, int32_t K, float* dimg, float* dfilt, cpcsv_stream_t stream);
/* elementwise tanh forward/backward on fp32 */
int cpcsv_tanh_fwd(const float* x, float* y, int64_t n, cpcsv_stream_t stream);
int cpcsv_tanh_bwd(const float* y, const float* dy, float* dx, int64_t n, cpcsv_stream_t stream);

/* final layer of D_GET_LOGITS (model.py:79-80): out = sigmoid(t * alpha + bias) where
 * t = features . weight_orig, alpha = 1/sigma (device scalars); and its backward
 * dz = dout * out * (1 - out), dt = dz * alpha. */
int cpcsv_affine_sigmoid_fwd(const float* t, const float* alpha, const float* bias, float* out,
                             int64_t n, cpcsv_stream_t stream);
int cpcsv_affine_sigmoid_bwd(const float* dout, const float* out, const float* alpha, float* dt,
                             float* dz, int64_t n, cpcsv_stream_t stream);

/* ---------------------------------------------------------------- spectral norm (legacy hook)
 * torch.nn.utils.spectral_norm, 1 power iteration, eps 1e-12 (model.py:5,19,79,502-510;
 * SURVEY.md Appendix A).  W is [R, C] row-major fp32 (= weight_orig.reshape(Cout, -1)).
 * Updates u [R], v [C] in place, writes sigma = u^T W v and inv_sigma. */
int cpcsv_spectral_sigma(const float* W, int32_t R, int32_t C, float* u, float* v,
                         int32_t do_power_iteration, float eps, float* sigma, float* inv_sigma,
                         float* scratch /* >= C + R floats */, cpcsv_stream_t stream);

/* backward through W_eff = W / sigma with sigma = u^T W v (u, v constants):
 *   dW = (G - (sum(G .* W) / sigma) u v^T) / sigma,   G = dL/dW_eff, all [R, C] fp32.
 * scratch: >= 1 float. */
int cpcsv_spectral_bwd(const float* G, const float* W, const float* u, const float* v,
                       const float* sigma, int32_t R, int32_t C, float* dW, float* scratch,
                       cpcsv_stream_t stream);
/* cpcsv_spectral_bwd with *dot = sum(G .* W) already known (cpcsv_unpack_conv_wgrad_dot):
 * dW = (G - (dot / sigma) u v^T) / sigma; G and dW may alias */
int cpcsv_spectral_bwd_apply(const float* G, const float* u, const float* v, const float* sigma,
                             const float* dot, int32_t R, int32_t C, float* dW, cpcsv_stream_t stream);


/* ------------------------------------------------------------------ optimiser (Adam)
 * optim.Adam(lr, betas=(0.5, 0.999)) of reference trainer.py:212-220, stepped at trainer.py:345-346
 * (discriminators) and trainer.py:416 (generator): fp32 Adam without weight decay, as multi-tensor
 * kernels FUSED with the re-layout of the updated weights into the 16-bit GEMM operand planes
 * (what cpcsv_pack_conv_weight / cpcsv_pack_matrix would otherwise redo after every step).
 * `step` (device float) counts optimiser steps; cpcsv_adam_tick advances it and writes
 * bc = { 1 / (1 - beta1^t), 1 / sqrt(1 - beta2^t) }; `lr` is a device scalar so a schedule
 * (trainer.py:447-456) acts on replayed CUDA graphs. */
typedef struct {
  const float* lr; /* device scalar */
  const float* bc; /* device [2], from cpcsv_adam_tick */
  double beta1, beta2, eps; /* doubles: 1 - beta2 is formed in double, as torch.optim.Adam does */
} cpcsv_adam_t;

typedef struct {
  float* p;
  const float* g;
  float* m; /* exp_avg */
  float* v; /* exp_avg_sq */
  int64_t n;
} cpcsv_adam_tensor_t;

/* one packed operand plane (pair) of a conv weight; kinds as cpcsv_pack_conv_weight */
typedef struct {
  int32_t kind, dtype, rows_pad, cols_pad;
  void* hi;
  void* lo; /* may be NULL */
} cpcsv_plane_t;

#define CPCSV_MAX_PLANES 6

int cpcsv_adam_tick(float* step, double beta1, double beta2, float* bc, cpcsv_stream_t stream);
/* plain parameters (BatchNorm affine, biases, GRU / Linear weights of the conditioning path) */
int cpcsv_adam_multi(const cpcsv_adam_tensor_t* tensors, int32_t count, const cpcsv_adam_t* hyper,
                     cpcsv_stream_t stream);
/* conv weight [Cout, Cin, kh, kw] (kh*kw <= 16): Adam step (skipped when g == NULL: pack only) and
 * every plane of `planes` rewritten from the updated values, padding included */
int cpcsv_adam_pack_conv(float* p, const float* g, float* m, float* v, int32_t Cout, int32_t Cin,
                         int32_t kh, int32_t kw, const cpcsv_adam_t* hyper, const cpcsv_plane_t* planes,
                         int32_t n_planes, cpcsv_stream_t stream);
/* fc / fc_seg weight [C*P, K] (model.py:260-263,285-288; P = 16 positions of the 4x4 map):
 * Adam step (g == NULL: pack only) + the NHWC-ordered planes: fwd16 fp16 [P*Cp, Kp], fwd_hi/lo
 * bf16 [P*Cp, Kp], bwd bf16 [Kp, P*Cp] (row j = c*P + pos -> j' = pos*Cp + c); any may be NULL */
int cpcsv_adam_pack_fc(float* p, const float* g, float* m, float* v, int32_t C, int32_t K, int32_t P,
                       int32_t Cp, int32_t Kp, const cpcsv_adam_t* hyper, void* fwd16, void* fwd_hi,
                       void* fwd_lo, void* bwd, cpcsv_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* CPCSV_H_ */
