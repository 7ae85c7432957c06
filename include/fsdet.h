/*
 * libfsdet.so — C ABI of the B200-native few-shot-detection training hot path.
 *
 * Drop-in boundary.  The reference (bingykang/Fewshot_Detection) reaches its
 * device code through torch-0.3.1 library calls made from
 * darknet_meta.py / dynamic_conv.py / region_loss.py; its only own FFI
 * precedent is layers/batchnorm/src/batchnorm.h:1-6 (plain C symbols, caller
 * allocates every output and workspace, launches on the current device).  This
 * header keeps that contract:
 *
 *   - plain C, raw device pointers + sizes, no torch types;
 *   - the caller owns all memory (outputs and workspaces are passed in); the
 *     library never allocates, frees or synchronises;
 *   - every function launches on `stream` (a cudaStream_t passed as void*) of the
 *     CURRENT device and returns immediately;
 *   - return value: 0 = ok, <0 = invalid argument (see fsdet_last_error()),
 *     >0 = cudaError_t of the failed launch;
 *   - re-entrant: no mutable global state - the only process-wide data are two
 *     driver entry points resolved once (thread-safe, immutable afterwards);
 *     one thread per GPU or one process per GPU are both fine.
 *
 * Layouts.  Activations inside the library are NHWC fp32: a 2-D array
 * [B*H*W pixels][ld] of which `C` channels starting at the given pointer are
 * used (ld >= C lets a layer write straight into a slice of a route/concat
 * buffer).  Convolution weights are OHWI ([Cout][kh*kw][Cin], i.e. torch
 * channels_last storage of the reference's OIHW nn.Conv2d.weight).  The
 * reference-facing tensors (input images, head output, loss targets) are NCHW
 * exactly as darknet_meta.Darknet.forward / RegionLossV2.forward exchange them.
 *
 * Each entry point cites the reference code it replaces (paths relative to
 * /root/reference).
 */
#ifndef FSDET_H_
#define FSDET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library info ----------------------------------------------------- */
int fsdet_version(void);
/* thread-local description of the last non-zero return value */
const char* fsdet_last_error(void);
/* compute capability the kernels were compiled for (100 = sm_100a) */
int fsdet_compiled_arch(void);

/* ---- layout conversion at the reference-facing boundary ---------------- */
/* [B,C0,H,W] (+ optional second tensor [B,C1,H,W], the support branch's
 * torch.cat([metax, mask], 1), darknet_meta.py:117-118) -> NHWC [B*H*W][ld],
 * channels C0+C1..Cpad-1 zero filled. */
int fsdet_nchw_to_nhwc(const float* in0, int C0, const float* in1, int C1, float* out, int ld, int Cpad,
                       int B, int HW, void* stream);
/* NHWC [B*HW][ld] (first C channels) (+ optional bias[C]) -> NCHW [B,C,HW] */
int fsdet_nhwc_to_nchw(const float* in, int ld, const float* bias, float* out, int B, int C, int HW, void* stream);

/* ---- convolution (nn.Conv2d stride 1, pad (k-1)/2; darknet_meta.py:219-259) */
/* Implicit GEMM  z[p][n] = sum_{tap,ci} x[p+tap][ci] * w[n][tap][ci] (+bias[n])
 * (+ previous z when accumulate != 0).  Used for forward (w = OHWI weights) and
 * for the input gradient (x = dz, w = fsdet_weight_flip_transpose(weights)).
 * stat_partial (optional): per-CTA column statistics for train-mode BatchNorm,
 * float [fsdet_conv_stat_rows(B*H*W)][4*Cout] = (sum | sum of squares | min | max).
 * Requires Cin % 4 == 0, ldx % 4 == 0, 16-byte aligned pointers. */
int fsdet_conv_fwd(const float* x, int ldx, const float* w, const float* bias, float* z, int ldz,
                   float* stat_partial, int B, int H, int W, int Cin, int Cout, int ksize, int accumulate,
                   void* stream);
int fsdet_conv_stat_rows(int npix);
/* Weight gradient dw[n][tap][ci] = sum_p dz[p][n] * x[p+tap][ci]  (OHWI).
 * workspace: float [fsdet_conv_wgrad_workspace_floats(...)] (split-K partials,
 * reduced in a fixed order: deterministic). */
int fsdet_conv_wgrad(const float* x, int ldx, const float* dz, int lddz, float* dw, float* workspace,
                     size_t workspace_floats, int B, int H, int W, int Cin, int Cout, int ksize, void* stream);
size_t fsdet_conv_wgrad_workspace_floats(int B, int H, int W, int Cin, int Cout, int ksize);
/* First layer, read straight from the reference-facing NCHW tensors (in0 [B,C0,H,W] and optionally in1
 * [B,C1,H,W] = the support branch's torch.cat([metax, mask], 1); C0+C1 <= 8; Cout <= 32; 3x3, pad 1):
 * forward z NHWC fp32 with weights zero-padded to [Cout][9][P]; weight gradient dw [Cout][9][P], its padding channels
 * written as zeros.  Channel pitch P = 4 when C0+C1 <= 4 (image + mask), 8 when C0+C1 is 5..8 (image + cropped object
 * [+ mask], metain_type 3 / 4).  HBM-bound kernels; workspace float [fsdet_conv_first_wgrad_workspace_floats_cin()]
 * (fsdet_conv_first_wgrad_workspace_floats() = the same for Cin <= 4).  The weight gradient stages x rows and dz rows
 * in shared memory: fsdet_conv_first_wgrad_supported(Cin, W) says whether they fit (8 channels: W <= 518). */
int fsdet_conv_first_fwd(const float* in0, int C0, const float* in1, int C1, const float* w_pad, float* z, int ldz,
                         int B, int H, int W, int Cout, void* stream);
/* The same convolution with the train-mode BatchNorm partial rows taken from the values in registers: stat_partial float
 * [fsdet_conv_first_stat_rows(B, H, W)][4*Cout] = (sum | sum of squares | min | max) per CTA - no fsdet_colstats pass. */
int fsdet_conv_first_stat_rows(int B, int H, int W);
int fsdet_conv_first_fwd_stats(const float* in0, int C0, const float* in1, int C1, const float* w_pad, float* z, int ldz,
                               int B, int H, int W, int Cout, float* stat_partial, void* stream);
int fsdet_conv_first_wgrad(const float* in0, int C0, const float* in1, int C1, const float* dz, int lddz, float* dw,
                           float* workspace, size_t workspace_floats, int B, int H, int W, int Cout, void* stream);
size_t fsdet_conv_first_wgrad_workspace_floats(int B, int H, int W, int Cout);
size_t fsdet_conv_first_wgrad_workspace_floats_cin(int B, int H, int W, int Cin, int Cout);
int fsdet_conv_first_wgrad_supported(int Cin, int W);
/* The same first block (conv 3x3 from <= 4 NCHW input channels into Cout <= 32 + train-mode BatchNorm + LeakyReLU +
 * MaxPool 2/2) WITHOUT storing its pre-BN output: every pass recomputes it from the input images with a tcgen05 GEMM
 * per 128-pixel tile (csrc/conv_first_tc.cuh).  Needs H % 8 == 0, W % 16 == 0 (fsdet_conv_first_tc_supported).
 * amax_x: device scalar >= max |input| (fsdet_amax over the input tensors).  w_pad4 as above.
 *   _stats      -> BatchNorm partial rows float [fsdet_conv_first_tc_rows(B,H,W)][4*Cout] for fsdet_bn_finalize
 *   _apply      -> leaky(z*scale+shift) max-pooled, as fp32 [B*(H/2)*(W/2)][ld_pool] and / or scaled fp16 hi/lo planes
 *                  [..][cpad] (cpad % 32 == 0, padding channels zero filled; amax_y from fsdet_bn_finalize)
 *   _bwd_reduce -> double [rows][3*Cout] = (sum du | sum du*xhat | max |du|) for fsdet_bn_bwd_finalize, du = dy_pool
 *                  routed to the first arg-max of each window (torch max_pool2d) times leaky'
 *   _bwd_wgrad  -> dw [Cout][9][4]: dz = scale*(du - c1 - xhat*c2) (coef = (c1 | c2) from fsdet_bn_bwd_finalize) is
 *                  formed tile by tile in shared memory and contracted with the im2col tile by a second GEMM; amax_dz
 *                  = the bound fsdet_bn_bwd_finalize writes; workspace float [fsdet_conv_first_tc_wgrad_workspace_floats] */
int fsdet_conv_first_tc_supported(int H, int W, int Cout);
int fsdet_conv_first_tc_rows(int B, int H, int W);
int fsdet_conv_first_tc_stats(const float* in0, int C0, const float* in1, int C1, const float* w_pad4, const float* amax_x,
                              float* stat_partial, int B, int H, int W, int Cout, void* stream);
int fsdet_conv_first_tc_apply(const float* in0, int C0, const float* in1, int C1, const float* w_pad4, const float* amax_x,
                              const float* scale, const float* shift, float slope, float* y_pool, int ld_pool, void* pool_hi,
                              void* pool_lo, int cpad, const float* amax_y, int B, int H, int W, int Cout, void* stream);
int fsdet_conv_first_tc_bwd_reduce(const float* in0, int C0, const float* in1, int C1, const float* w_pad4, const float* amax_x,
                                   const float* scale, const float* shift, const float* mean, const float* invstd, float slope,
                                   const float* dy_pool, int ld_dyp, double* partial, int B, int H, int W, int Cout, void* stream);
size_t fsdet_conv_first_tc_wgrad_workspace_floats(int B, int H, int W);
int fsdet_conv_first_tc_bwd_wgrad(const float* in0, int C0, const float* in1, int C1, const float* w_pad4, const float* amax_x,
                                  const float* scale, const float* shift, const float* mean, const float* invstd,
                                  const double* coef, float slope, const float* dy_pool, int ld_dyp, const float* amax_dz, float* dw,
                                  float* workspace, size_t workspace_floats, int B, int H, int W, int Cout, void* stream);
/* wt[ci][kk-1-tap][co] = w[co][tap][ci]  (weights for the input-gradient conv) */
int fsdet_weight_flip_transpose(const float* w, float* wt, int Cout, int kk, int Cin, void* stream);
/* copy [rows][cin] -> [rows][cout] channel-padded / -cropped (zero fill) */
int fsdet_pad_channels(const float* in, int cin, float* out, int cout, size_t rows, void* stream);

/* ---- tensor-core convolution (tcgen05 + TMA im2col), csrc/conv_tc.cu ---- */
/* Same contraction as fsdet_conv_fwd for layers with Cin % 32 == 0, Cout % 4 == 0
 * (fsdet_conv_tc_supported); `cpitch` >= Cin is the channel pitch of the planes
 * (activation rows and the weights' [tap][channel] axis), so 32-channel tensors
 * stored in 64-channel-padded planes are read without touching the padding.
 * Operands are fp16 hi/lo planes (fsdet_amax + fsdet_split_f16, or written
 * directly by the producing BN / weight-preparation kernels): the tensor is
 * scaled by the power of two that maps its absolute maximum into [512, 1024),
 * hi = fp16(s*x), lo = fp16(s*x - hi).
 * `mode`: bits 0-1 select the operand terms added to hi*hi -
 *     bit 0: x_lo * w_hi (x exact to 22 bits), bit 1: x_hi * w_lo (w exact);
 *     3 = fp32-grade (reproduces the fp32 reference incl. its max-pool arg-max
 *     decisions), 0 = plain fp16 x fp16 -> fp32.  Planes that are not used may be
 *     NULL.  Bit 4 (16): persistent tile loop for short-K layers (one CTA per
 *     SM, double-buffered TMEM accumulators).  Bit 5 (32): thread-block clusters
 *     of two CTAs that share the weight tile through TMA multicast (ignored in
 *     persistent mode and for single-tile problems).  Bit 6 (64): never take the
 *     halo-tile kernel.  By default (bits 4-6 clear, mode 3) the 3x3 layers with
 *     Cin in {32, 64, 128}, Cout <= 128, W % 8 == 0 and enough 8 x 16 pixel tiles
 *     run the halo-tile kernel (csrc/conv_halo_kernels.cuh: the input tile is
 *     fetched once with its halo for all nine taps instead of once per tap - those
 *     layers are L2-bandwidth bound otherwise); fsdet_conv_tc_uses_halo tells.
 *     Bit 7 (128): issue x_hi*w_hi and x_hi*w_lo as two MMAs.  By default the
 *     mode-3 kernels with one hi accumulator issue them as ONE MMA of width
 *     2*BN (the lo weight plane follows the hi plane in shared memory, the lo
 *     accumulator follows the hi accumulator in TMEM): same products, two
 *     tcgen05.mma per K step instead of three.
 * x_hi/x_lo dense NHWC [B*H*W][cpitch] fp16, w_hi/w_lo [Cout][k*k*cpitch] fp16,
 * amax_x / amax_w: device floats holding the tensors' absolute maxima (NULL =
 * planes are unscaled).  Output fp32 z[p][n] (+ previous z when accumulate
 * != 0).
 * stat_partial (optional, accumulate == 0 only): train-mode BatchNorm partial
 * rows float [fsdet_conv_tc_stat_rows(...)][4*Cout] = (sum | sum of squares |
 * min | max) per CTA, taken from the output tile in the epilogue (no separate
 * pass over z); the layout fsdet_bn_finalize reads. */
int fsdet_conv_tc_supported(int Cin, int Cout, int ksize);
int fsdet_conv_tc_stat_rows(int B, int H, int W, int Cin, int Cout, int ksize, int mode);
int fsdet_conv_tc_uses_halo(int B, int H, int W, int Cin, int Cout, int ksize, int mode);
int fsdet_conv_tc_fwd(const void* x_hi, const void* x_lo, const void* w_hi, const void* w_lo, const float* amax_x,
                      const float* amax_w, float* z, int ldz, int B, int H, int W, int Cin, int cpitch, int Cout,
                      int ksize, int accumulate, int mode, float* stat_partial, void* stream);
/* Weight gradient on the tensor cores (pixels are the GEMM K dimension; both
 * operands are consumed MN-major straight from the NHWC planes).  Needs
 * Cin % 64 == 0 and Cout % 64 == 0.  dw [Cout][k*k][Cin] fp32 (OHWI);
 * workspace float [fsdet_conv_tc_wgrad_workspace_floats(...)] for the split-K
 * partials (reduced in a fixed order).  `mode` bits 0-1 as above with
 * bit 0: dz_lo * x_hi, bit 1: dz_hi * x_lo. */
int fsdet_conv_tc_wgrad_supported(int Cin, int Cout, int ksize);
size_t fsdet_conv_tc_wgrad_workspace_floats(int B, int H, int W, int Cin, int Cout, int ksize, int mode);
int fsdet_conv_tc_wgrad(const void* x_hi, const void* x_lo, const void* dz_hi, const void* dz_lo, const float* amax_x,
                        const float* amax_dz, float* dw, float* workspace, size_t workspace_floats, int B, int H,
                        int W, int Cin, int Cout, int ksize, int mode, void* stream);
/* All weight operands of a network for the tensor-core convolutions in two launches (csrc/weights.cu): absolute
 * maxima, then the scaled fp16 (hi, lo) planes of every layer in the forward order [Cout][tap*fwd_pitch + ci] and -
 * when bwd_hi != NULL - flip-transposed for the input-gradient GEMM [Cin][(kk-1-tap)*bwd_pitch + co].
 * descs_dev: device array of n_layers descriptors; tiles_dev: device int32 pairs (layer, tile) with tile in
 * [0, kk*tiles_co*tiles_ci) enumerating the 32x32 (Cout x Cin) tiles of every filter tap; amax_all: device float
 * [n_layers] (desc.amax points into it).  The planes' channel padding (pitch > channels) is never written: allocate
 * them zeroed once.  Replaces fsdet_amax + fsdet_split_f16 + fsdet_weight_flip_transpose + fsdet_split_f16 per layer. */
typedef struct fsdet_weight_desc {
    const float* w;      /* OHWI fp32 [Cout][kk][Cin] (torch channels_last storage of nn.Conv2d.weight) */
    void* fwd_hi;        /* fp16 [Cout][kk*fwd_pitch] or NULL */
    void* fwd_lo;
    void* bwd_hi;        /* fp16 [Cin][kk*bwd_pitch] or NULL */
    void* bwd_lo;
    float* amax;         /* device scalar, written by the first pass */
    int32_t Cout, kk, Cin, fwd_pitch, bwd_pitch, tiles_ci, tiles_co, reserved;
} fsdet_weight_desc;
int fsdet_weight_prep(const fsdet_weight_desc* descs_dev, const int32_t* tiles_dev, int n_tiles, float* amax_all,
                      int n_layers, void* stream);
/* absolute maximum of fp32 [rows][ld] (first C columns) -> *amax_out (device float) */
int fsdet_amax(const float* src, int ld, int C, size_t rows, float* amax_out, void* stream);
/* the same without resetting the destination first: *amax_inout = max(*amax_inout, max |src|) */
int fsdet_amax_acc(const float* src, int ld, int C, size_t rows, float* amax_inout, void* stream);
/* fp32 [rows][ld] (first C columns) -> two dense fp16 planes [rows][Cpad] of the
 * tensor scaled as described above (amax NULL: no scaling); columns C..Cpad-1
 * are zero (lets 32-channel layers use the 64-channel K tiles) */
int fsdet_split_f16(const float* src, int ld, int C, int Cpad, size_t rows, const float* amax, void* hi, void* lo,
                    void* stream);
/* per-strip column statistics of z: float [fsdet_colstats_rows(npix)][4*C] = (sum | sum of squares | min | max) */
int fsdet_colstats(const float* z, int ld, size_t npix, int C, float* partial, void* stream);
int fsdet_colstats_rows(size_t npix);
/* test hook: one im2col TMA tile (128 pixels x 64 channels of filter tap `tap`,
 * starting at output pixel m0, channel c0) un-swizzled to out_tile [128][64] bf16 */
int fsdet_debug_im2col_tile(const void* x_plane, int B, int H, int W, int C, int ksize, long long m0, int c0, int tap,
                            void* out_tile, void* stream);

/* ---- BatchNorm2d(train/eval) + LeakyReLU(0.1) + MaxPool2d(2,2) -------- */
/* nn.BatchNorm2d defaults (darknet_meta.py:247): eps 1e-5, momentum 0.1, biased
 * batch variance for normalisation, unbiased for running_var.
 * Reduces the conv partial rows float [nparts][4*C] = (sum | sum of squares | min
 * | max per channel; written by fsdet_conv_fwd or fsdet_colstats; the buffer
 * must have fsdet_bn_stat_scratch_rows() further rows of scratch); writes
 * mean/invstd (saved for backward) and the fused per-channel scale/shift; updates
 * running stats when training != 0.  amax_y (optional device float): exact
 * absolute maximum of y = leaky(z*scale+shift, slope) over the tensor, derived
 * from the per-channel range of z (scale of the fp16 planes of y).  In eval mode
 * (training == 0) scale/shift come from the running statistics, stat_partial is
 * ignored and amax_y is not written.  xhat_absmax (optional, [C]): max over
 * the batch of |(z - mean) * invstd| per channel (used by the backward pass
 * to bound max|dz|). */
int fsdet_bn_finalize(const float* stat_partial, int nparts, double count, const float* gamma, const float* beta,
                      float* running_mean, float* running_var, float momentum, float eps, float* mean,
                      float* invstd, float* scale, float* shift, float slope, float* amax_y, float* xhat_absmax,
                      int C, int training, void* stream);
int fsdet_bn_stat_scratch_rows(void);
/* y = leaky(z*scale+shift, slope), written in one pass as any subset of: fp32
 * full resolution (y_full), fp32 MaxPool2d(2,2) (floor) output (y_pool), and the
 * fp16 hi/lo planes [pixels][Cpad] of either (for the tensor-core convolutions;
 * scaled by the power of two derived from *amax, channels C..Cpad-1 zero). */
int fsdet_bn_act_fwd(const float* z, int ldz, const float* scale, const float* shift, float slope, float* y_full,
                     int ld_full, float* y_pool, int ld_pool, void* full_hi, void* full_lo, void* pool_hi,
                     void* pool_lo, int Cpad, const float* amax, int B, int H, int W, int C, void* stream);
/* Backward of the block above.  dy_full / dy_pool: gradients w.r.t. the two
 * outputs (either may be NULL).  Pass 1 reduces, per CTA row,
 * [sum(du) | sum(du*xhat) | max|du|] into partials double
 * [fsdet_bn_bwd_rows(B,H,W) + 1][3*C] (the extra row receives the totals in
 * fsdet_bn_bwd_finalize); pass 2 (after fsdet_bn_bwd_finalize) writes dz.
 * The projection dz = scale*(du - mean(du) - xhat*mean(du*xhat)) cancels
 * heavily and float32 sums lose 2-3 digits there (torch's CPU kernel uses double
 * accumulators for the same reason): sums are accumulated to double accuracy
 * (compensated fp32 per thread, double across threads), coefficients are
 * double, and the apply pass subtracts mean(du) as a (hi, lo) float pair.
 * With has_bn == 0 (conv + bias + act): xhat terms are skipped, dbeta = bias
 * gradient, dz = du. */
int fsdet_bn_act_bwd_reduce(const float* z, int ldz, const float* dy_full, int ld_dyf, const float* dy_pool,
                            int ld_dyp, const float* scale, const float* shift, const float* mean,
                            const float* invstd, float slope, double* partial, int B, int H, int W, int C,
                            int has_bn, void* stream);
int fsdet_bn_bwd_rows(int B, int H, int W);
/* dgamma, dbeta, the two per-channel coefficients used by the apply pass and
 * (optional) *amax_bound >= max|dz|, from |dz| <= |scale|*(max|du| + |c1| +
 * max|xhat|*|c2|) with max|xhat| = xhat_absmax from fsdet_bn_finalize: the
 * power-of-two scale of dz's fp16 planes. */
int fsdet_bn_bwd_finalize(const double* partial, int nparts, double count, const float* gamma, const float* invstd,
                          const float* xhat_absmax, float* dgamma, float* dbeta, double* coef /* [2*C] */,
                          float* amax_bound, int C, int has_bn, void* stream);
/* dz as fp32 (dz, may be NULL) and/or directly as the scaled fp16 hi/lo planes
 * [pixels][cpad] read by the tensor-core GEMMs (dz_hi/dz_lo, may be NULL;
 * cpad == C; scaled by the power of two derived from *amax, which must bound
 * max|dz| - use fsdet_bn_bwd_finalize's amax_bound). */
int fsdet_bn_act_bwd_apply(const float* z, int ldz, const float* dy_full, int ld_dyf, const float* dy_pool,
                           int ld_dyp, const float* scale, const float* shift, const float* mean,
                           const float* invstd, const double* coef, float slope, float* dz, int lddz, void* dz_hi,
                           void* dz_lo, int cpad, const float* amax, int B, int H, int W, int C, int has_bn,
                           void* stream);

/* ---- stand-alone pooling / reorg / route (darknet_meta.py:47-74,157-171) */
/* size 2; stride 2 (floor) or stride 1 with replicate pad right/bottom
 * (MaxPoolStride1, darknet_meta.py:47-53) */
int fsdet_maxpool_fwd(const float* x, int ldx, float* y, int ldy, int B, int H, int W, int C, int stride, void* stream);
int fsdet_maxpool_bwd(const float* x, int ldx, const float* dy, int lddy, float* dx, int lddx, int B, int H, int W,
                      int C, int stride, void* stream);
/* Reorg(2): out[b,(i*2+j)*C+c,h,w] = x[b,c,2h+i,2w+j] (darknet_meta.py:55-74) */
int fsdet_reorg_fwd(const float* x, int ldx, float* y, int ldy, int B, int H, int W, int C, void* stream);
int fsdet_reorg_bwd(const float* dy, int lddy, float* dx, int lddx, int B, int H, int W, int C, void* stream);
/* GlobalMaxPool2d (pooling.py:8-27): y[n][c] = max_p x[n][p][c]; argmax saved */
int fsdet_globalmax_fwd(const float* x, int ldx, float* y, int32_t* argmax, int N, int HW, int C, void* stream);
int fsdet_globalmax_bwd(const float* dy, const int32_t* argmax, float* dx, int lddx, int N, int HW, int C, void* stream);
/* dst[p][0..C) = (accumulate ? dst : 0) + src[p][0..C)   (route/concat, grad sum) */
int fsdet_copy_channels(const float* src, int ldsrc, float* dst, int lddst, size_t npix, int C, int accumulate,
                        void* stream);

/* ---- per-class reweighting fused into the 1x1 detection conv ----------- */
/* dynamic_conv.DynamicConv2d.forward (dynamic_conv.py:125-164) followed by the
 * head nn.Conv2d(1024, 30, 1):  out[b*n_cls+c] = (W (.) rw[c]) x[b] + bias.
 * weff[(c*O+o)][k] = W[o][k]*rw[c][k]  (rows padded to Npad with zeros),
 * bias_eff[c*O+o] = bias[o]. The GEMM itself runs through fsdet_conv_fwd. */
int fsdet_head_weff(const float* W, const float* bias, const float* rw, float* weff, float* bias_eff, int n_cls,
                    int O, int K, int Npad, void* stream);
/* dW[o][k] = sum_c dweff[c*O+o][k]*rw[c][k]; drw[c][k] = sum_o dweff[c*O+o][k]*W[o][k] */
int fsdet_head_param_grads(const float* dweff, const float* W, const float* rw, float* dW, float* drw, int n_cls,
                           int O, int K, void* stream);
/* column sums of an NHWC matrix folded over classes: dbias[o] = sum_{p,c} d[p][c*O+o] */
int fsdet_head_bias_grad(const float* d, int ld, float* dbias, float* workspace /* [rows][n_cls*O] */,
                         size_t npix, int n_cls, int O, void* stream);
size_t fsdet_head_bias_grad_workspace_floats(size_t npix, int n_cls, int O);

/* ---- region loss (region_loss.py) -------------------------------------- */
/* RegionLoss(V2).forward prologue, region_loss.py:256-298: sigmoid / exp decode of the kept rows into
 * pred_boxes float32 [nB*A*H*W][4] in grid units.  inds (optional) = kept output rows (neg_filter).
 * nB_dev (optional, also below): device int32 holding the number of LIVE slots when the launch is frozen at a
 * capacity of nB rows (CUDA-graph replay: neg_filter keeps a different number of rows every step). */
int fsdet_region_decode(const float* output, const int32_t* inds, int nB, const int32_t* nB_dev, int A, int nC, int H,
                        int W, const float* anchors_f32 /* [2A] */, float* pred_boxes, void* stream);
/* build_targets, region_loss.py:37-132 (+ utils.bbox_ious / bbox_iou,
 * utils.py:21-83).  target: float64 [nB][250] rows already filtered, or - when
 * `inds` is given - the FULL label matrix, of which slot b reads row inds[b].  Outputs:
 * nine float32 [nB][A][H][W] tensors and counters int32[4] = {nGT, nCorrect,
 * n_degenerate (GT with w or h == 0: the reference raises there), 0}.
 * Index/mask outputs are bit-exact w.r.t. the reference; phase-1 IoUs are
 * computed in float32 with the reference's operation order and no FMA
 * contraction, phase 2 in float64. */
int fsdet_build_targets(const float* pred_boxes, const double* target, const double* anchors_f64 /* [2A] */,
                        int nB, int A, int H, int W, int max_boxes, float noobject_scale, float object_scale,
                        float sil_thresh, long long seen, float* coord_mask, float* conf_mask, float* cls_mask,
                        float* tx, float* ty, float* tw, float* th, float* tconf, float* tcls, int32_t* counters,
                        const int32_t* inds, const int32_t* nB_dev, void* stream);
/* Loss terms + gradient w.r.t. the raw head output (region_loss.py:303-345).
 * mode 0 = RegionLossV2 (softmax across the cs class rows of each image),
 * mode 1 = RegionLoss (softmax across nC channels; tcls zeroed if metayolo).
 * img_start[bs+1] = prefix of kept rows per image (V2).
 * losses: double[8] = {x,y,w,h,conf,cls,total,nProposals}
 * accumulated with atomics in double (zeroed by this call's first kernel). */
int fsdet_region_loss_grad(const float* output, float* grad_output, const int32_t* inds, const int32_t* nB_dev,
                           const int32_t* img_start, int rows_total, int nB, int bs, int cs, int A, int nC, int H,
                           int W, const float* coord_mask, const float* conf_mask, const float* cls_mask,
                           const float* tx, const float* ty, const float* tw, const float* th, const float* tconf,
                           const float* tcls, float coord_scale, float class_scale, int mode, int metayolo,
                           double* losses, void* stream);

/* ---- optimiser (optim.SGD as configured in train_meta.py:143-147) ------ */
/* One launch over a table of tensors: d = g + wd*p; m = first ? d : mom*m + (1-damp)*d;
 * p -= lr*m.  ptr tables live in device memory: params/grads/moms [n] pointers,
 * sizes [n] element counts, chunk table built by the caller (see optim.py).
 * hyper_dev (optional): device float[4] = {lr, momentum, dampening, weight_decay}
 * overriding the scalar arguments, so that a CUDA-graph-captured step can follow
 * the driver's learning-rate schedule (train_meta.py:150-163). */
int fsdet_sgd_step(float* const* params, const float* const* grads, float* const* moms, const long long* sizes,
                   const int32_t* chunk_tensor, const long long* chunk_offset, int n_chunks, int chunk_elems,
                   float lr, float momentum, float dampening, float weight_decay, int first_step,
                   const float* hyper_dev, void* stream);

/* ---- evaluation: detection decode + NMS (SURVEY.md 8f row 1) ------------- */
/* utils.get_region_boxes (utils.py:112-193; v2 = 0, n_models = 1) and utils.get_region_boxes_v2 (utils.py:195-290;
 * v2 = 1: rows are (image, class) pairs, image-major, and the class score is the softmax ACROSS the n_models rows of
 * an image).  output: float32 [N][A*(5+nC)][H][W] (the head output).  For every row n the anchor-cells with
 * (only_objectness ? det_conf : det_conf*cls_max_conf) > conf_thresh (float64 test, as the reference's Python-float
 * arithmetic) are written in the reference's loop order (cy, cx, anchor) to cand[n][0..count[n])[8] =
 * {xs, ys, ws, hs (grid units, float32), det_conf, cls_max_conf, (int32 bits) cls_max_id, (int32 bits) a*H*W + cell};
 * capacity per row = A*H*W.  cls_dense (optional, float32 [N*A*H*W][nC]) receives the softmax scores that the
 * reference's `validation=True` branch reads (utils.py:176-181).  No device->host copy, no synchronisation. */
int fsdet_region_detect(const float* output, const float* anchors_f32 /* [2A] */, int N, int A, int nC, int H, int W,
                        int n_models, int v2, int only_objectness, double conf_thresh, float* cand, int32_t* count,
                        float* cls_dense, void* stream);
/* utils.nms (utils.py:85-104) for all N rows at once: boxes normalised in float64 (x/W, y/H, w/W, h/H), sorted by
 * float32(1 - det_conf) ascending (ties: candidate order), greedy suppression with the float64 utils.bbox_iou
 * (utils.py:21-52) > nms_thresh.  keep[n][0..keep_count[n]) = candidate slots of the survivors in that order.
 * cap = candidates per row of `cand` (<= 4096). */
int fsdet_nms(const float* cand, const int32_t* count, int N, int cap, int H, int W, double nms_thresh, int32_t* keep,
              int32_t* keep_count, void* stream);
/* Same for rows of already-normalised float64 boxes [N][cap][5] = {x, y, w, h, det_conf}: the list-of-lists form in
 * which utils.nms (utils.py:85) receives boxes from any caller (e.g. utils.do_detect, utils.py:410-458). */
int fsdet_nms_boxes64(const double* boxes, const int32_t* count, int N, int cap, double nms_thresh, int32_t* keep,
                      int32_t* keep_count, void* stream);
/* Running mean of the support net's reweighting vectors per class, valid_ensemble.py:86-100:
 * for i in 0..n-1: c = ids[i]; enews[c] = enews[c]*cnt[c]/(cnt[c]+1) + dw[i]/(cnt[c]+1); cnt[c] += 1 (float32, the
 * reference's operation order).  enews float32 [n_cls][C] (zero before the first call), dw float32 [n][C];
 * cnt_in / cnt_out int32 [n_cls] must be different buffers. */
int fsdet_rw_running_mean(float* enews, const int32_t* cnt_in, int32_t* cnt_out, const float* dw, const int32_t* ids,
                          int n, int n_cls, int C, void* stream);

/* ---- training-input augmentation (SURVEY.md 8f row 3) ---------------------- */
/* image.data_augmentation (image.py:52-87: crop with zero fill, PIL resize, horizontal flip, HSV jitter through
 * image.distort_image :19-37) + transforms.ToTensor for n images in one launch pair.
 *   src    device array of n pointers to decoded uint8 RGB images, HWC
 *   geom   int32 [n][8] = {ow, oh, pleft, ptop, crop_w, crop_h, flip, distort}; the reference's crop box is
 *          (pleft, ptop, pleft + swidth - 1, ptop + sheight - 1), i.e. crop_w = swidth - 1 (image.py:72)
 *   color  float64 [n][3] = {dhue, dsat, dexp} (image.py:45-50)
 *   filter 0 = PIL NEAREST, 3 = PIL BICUBIC (the default of `Image.resize` before / since Pillow 7)
 *   kmax   bound on the resampling taps per output coordinate: >= 2*ceil(2*max(crop/out, 1)) + 1
 *   out    float32 [n][3][H][W] = the uint8 result / 255; out_u8 (optional) uint8 [n][H][W][3] = that uint8 result
 *   status int32[1]: 0, or 1 + index of an image whose taps did not fit kmax / whose crop is empty
 * Bit-identical to Pillow's uint8 pipeline (integer resampling with 22-bit coefficients and a rounding after each
 * pass; Convert.c colour conversions; `point` tables rounded half-to-even). */
size_t fsdet_augment_workspace_bytes(int n, int W, int H, int kmax);
int fsdet_augment_batch(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W, int H,
                        int kmax, int filter, void* workspace, size_t workspace_bytes, float* out, uint8_t* out_u8,
                        int32_t* status, void* stream);
/* The same with image i written at out + i * out_pitch floats (out_pitch >= 3*H*W), so that several launches can fill
 * the channel groups of one [n][C][H][W] tensor.  fsdet_augment_batch = out_pitch 3*H*W.  The cropped-object channels
 * of metain_type 3 / 4 (dataset.py:378-398, `img.crop(rect).resize(img.size)`) are a second launch over the first
 * launch's out_u8 with geom {W, H, x1, y1, x2 - x1, y2 - y1, 0, 0}, into channels 3..5 of a 6-channel tensor. */
int fsdet_augment_batch_pitched(const uint8_t* const* src, const int32_t* geom, const double* color, int n, int W, int H,
                                int kmax, int filter, void* workspace, size_t workspace_bytes, float* out, size_t out_pitch,
                                uint8_t* out_u8, int32_t* status, void* stream);
/* dataset.MetaDataset.get_img_mask (dataset.py:378-398): out float32 [n][H][W] = 1 inside rects[i] = {x1, y1, x2, y2}
 * (half-open, already rounded and clamped by the caller as the reference does), else 0. */
int fsdet_box_masks(const int32_t* rects, int n, int H, int W, float* out, void* stream);

/* ---- misc --------------------------------------------------------------- */
int fsdet_fill(float* p, float v, size_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FSDET_H_ */
