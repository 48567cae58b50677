/*
 * mpgan.h -- C ABI of libmpgan_sm100.so: the B200 (sm_100a) kernels behind the GAN hot path of
 * mbrzus/Cross-Modality-Minipig-Gan.
 *
 * The reference has no FFI seam for this path: its arithmetic is PyTorch ops called from plain Python
 * classes (SURVEY.md section 8b).  Each entry point below replaces the torch op(s) named in its comment
 * (file:line into /root/reference).  Conventions:
 *   - extern "C", plain pointers and sizes only; the caller owns every buffer (device memory unless noted).
 *   - activations are channels-last: (N, [D,] H, W, C) with a pixel stride `ld*` in elements (>= C), so a
 *     tensor may be a channel slice of a wider concat buffer.
 *   - conv weights are "OTI": [Cy][tap][Cx] (taps in (kd,kh,kw) order) for the underlying convolution
 *     X-grid -> Y-grid; a ConvTranspose is the same weight used in the Y -> X direction.
 *   - dtype: MPGAN_F32 or MPGAN_BF16 for activations/weights; statistics, losses, master weights and
 *     gradients of parameters are always fp32 (batch-norm sums fp64).
 *   - every call is asynchronous on `stream` (a cudaStream_t), never synchronises or allocates, and is
 *     CUDA-graph-capture safe.  Return 0 on success; <0 on error, text via mpgan_last_error().
 *   - no CPU fallback exists: on a machine without a B200 the compute entry points fail with MPGAN_ERR_CUDA.
 */
#ifndef MPGAN_H_
#define MPGAN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPGAN_VERSION 100

enum { MPGAN_OK = 0, MPGAN_ERR_SHAPE = -1, MPGAN_ERR_UNSUPPORTED = -2, MPGAN_ERR_CUDA = -3 };
enum { MPGAN_F32 = 0, MPGAN_BF16 = 1 };
enum { MPGAN_ACT_NONE = 0, MPGAN_ACT_PRELU = 1, MPGAN_ACT_LEAKY = 2, MPGAN_ACT_TANH = 3 };

/* Geometry of the underlying convolution X-grid -> Y-grid (y = x*stride - pad + r). rank 2 uses index 1,2 of
 * the 3-vectors (index 0: size 1, k 1, stride 1, pad 0). */
typedef struct {
  int32_t rank;       /* 2 or 3 spatial dims */
  int32_t n;          /* batch */
  int32_t xs[3];      /* X-grid spatial extent (D,H,W) */
  int32_t ys[3];      /* Y-grid spatial extent */
  int32_t cx, cy;     /* channels on the X / Y side */
  int32_t k[3], stride[3], pad[3];
} MpganConvGeom;

int mpgan_version(void);
const char* mpgan_last_error(void);
/* 1 if a CUDA device of compute capability 10.x is usable by this process, else 0 (never raises). */
int mpgan_device_ok(void);

/* ---- convolution, generic CUDA-core path (any channel count, rank 2/3, f32 or bf16 storage, fp32 accumulate) ----
 * nn.Conv3d/Conv2d forward  (GAN_final.py:167-189, MONAI Convolution via GAN_final.py:106-114)  = fprop
 * nn.ConvTranspose forward  (MONAI up path)                                                       = bprop
 * and their data gradients (torch autograd's convolution_backward) the other way round.
 * `w` is OTI [cy][taps][cx] in `dtype`; bias fp32 [channels of the output side] or NULL. */
int mpgan_conv_fprop(const MpganConvGeom* g, int dtype, const void* x, int64_t ldx, const void* w,
                     const float* bias, void* y, int64_t ldy, void* stream);
int mpgan_conv_bprop(const MpganConvGeom* g, int dtype, const void* y, int64_t ldy, const void* w,
                     const float* bias, void* x, int64_t ldx, void* stream);
/* dw[cy][taps][cx] += sum_pixels y (x) x   (fp32, accumulates: the caller zeroes);  weight gradient of both
 * Conv and ConvTranspose. */
int mpgan_conv_wgrad(const MpganConvGeom* g, int dtype, const void* x, int64_t ldx, const void* y, int64_t ldy,
                     float* dw, void* stream);

/* ---- convolution, tcgen05 path (bf16 operands, fp32 TMEM accumulators, TMA-staged NHWC tiles; rank 2) ----
 * Same contracts as above with dtype == BF16.  Requirements: cx, cy multiples of 16 (>= 16).
 * w_f is OTI [cy][taps][cx] bf16 (used by fprop); w_b is its transpose [cx][taps][cy] bf16 (used by bprop).
 * Optional fused epilogue: bias add and per-channel batch-norm partial sums (sum, sum of squares of the
 * stored bf16 values) accumulated into stats[2*C] (fp64, caller zeroes) when stats != NULL. */
int mpgan_tc_supported(const MpganConvGeom* g, int direction /*0 fprop,1 bprop,2 wgrad*/);
int mpgan_tc_conv_fprop(const MpganConvGeom* g, const void* x, int64_t ldx, const void* w_f, const float* bias,
                        void* y, int64_t ldy, double* stats, void* stream);
int mpgan_tc_conv_bprop(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b, const float* bias,
                        void* x, int64_t ldx, double* stats, void* stream);
/* same, with a bf16 tensor `res` (pixel stride ldres, the X grid) added to the result before rounding: fuses the
 * gradient accumulation of residual / skip branches (dx = dgrad(dy) + res) into the convolution's epilogue */
/* inference-mode fused layer (BatchNorm folded into w / bias by the caller):  out = prelu(conv(in, w) + bias) + res
 * direction 0: convolution X -> Y with w = [cy][taps][cx]; direction 1: transposed convolution Y -> X with the
 * transposed weights [cx][taps][cy].  slope: device scalar (PReLU weight) or NULL (no activation); res optional. */
int mpgan_tc_conv_act(const MpganConvGeom* g, int direction, const void* in, int64_t ldi, const void* w,
                      const float* bias, const float* slope, const void* res, int64_t ldres, void* out, int64_t ldo,
                      void* stream);
/* ConvTranspose(cy -> 1, k3 s2 p1 op1) forward == data gradient of a one-input-channel stride-2 3x3 convolution, through
 * the halo tcgen05 kernel in pixel-shuffle mode: w = the layer's bf16 [cy][9] weight, x = (n, 2*yh, 2*yw) one channel,
 * stats (optional) = fp64 {sum, sum of squares} of the stored values (fused BatchNorm(1) statistics). */
int mpgan_tc_convt_to1(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w, const float* bias, void* x,
                       double* stats, void* stream);
/* data gradient of a one-input-channel stride-1 3x3 layer (cx == 1; dY has cy in {16,32,64,128} channels) through the
 * halo-resident tcgen05 kernel: w_b16 = bf16 [16][9][cy], row 0 the layer's transposed weights, rows 1..15 zero;
 * x: (n, xh, xw) one channel, pixel stride ldx; res (optional, same layout, stride ldres) is added. */
int mpgan_tc_conv_bprop_c1out(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b16, void* x,
                              int64_t ldx, const void* res, int64_t ldres, void* stream);
int mpgan_tc_conv_bprop_res(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b, const float* bias,
                            void* x, int64_t ldx, const void* res, int64_t ldres, double* stats, void* stream);
/* workspace_bytes from mpgan_tc_conv_wgrad_workspace(); dw accumulates (fp32 [cy][taps][cx]). */
size_t mpgan_tc_conv_wgrad_workspace(const MpganConvGeom* g);
int mpgan_tc_conv_wgrad(const MpganConvGeom* g, const void* x, int64_t ldx, const void* y, int64_t ldy, float* dw,
                        void* workspace, size_t workspace_bytes, void* stream);
/* ---- convolution, one-channel edge layers (SURVEY.md K6): bandwidth-bound direct kernels, rank 2/3, f32 or bf16 ----
 * fprop with cy == 1 or (rank 2, 3x3) cx == 1 (G's 1->16 and D's 1->64 first convolutions), bprop with cx == 1 (ConvTranspose 32->1
 * forward, data gradient of the 1->16 / 1->64 first convolutions), wgrad with cx == 1.  Same contracts as the generic
 * entry points; mpgan_c1_supported() says whether a (geometry, direction) is covered. */
int mpgan_c1_supported(const MpganConvGeom* g, int direction /*0 fprop,1 bprop,2 wgrad*/);
int mpgan_c1_conv_fprop(const MpganConvGeom* g, int dtype, const void* x, int64_t ldx, const void* w,
                        const float* bias, void* y, int64_t ldy, double* stats /* nullable: BN sums of y */,
                        void* stream);
/* inference fusion of a one-input-channel layer: y = prelu(conv(x, w) + bias), BatchNorm folded into (w, bias) by the caller
 * (MONAI Convolution in model.eval(), inferrence.py:107-109); returns -2 when the run-based kernel does not cover the layer */
int mpgan_c1_conv_act(const MpganConvGeom* g, int dtype, const void* x, int64_t ldx, const void* w, const float* bias,
                      const float* slope, void* y, int64_t ldy, void* stream);
int mpgan_c1_conv_bprop(const MpganConvGeom* g, int dtype, const void* y, int64_t ldy, const void* w,
                        const float* bias, void* x, int64_t ldx, double* stats /* nullable: BN sums of x */,
                        void* stream);
int mpgan_c1_conv_wgrad(const MpganConvGeom* g, int dtype, const void* x, int64_t ldx, const void* y, int64_t ldy,
                        float* dw, void* stream);

/* ---- batch norm (nn.BatchNorm3d, GAN_final.py:170-188; MONAI norm=BATCH) + activation, fused ----
 * stats: per-channel sum / sum-of-squares in fp64 (accumulates; caller zeroes). */
int mpgan_bn_stats(int dtype, const void* x, int64_t ldx, int64_t pixels, int32_t c, double* stats, void* stream);
/* training: batch mean / biased var -> scale=gamma*invstd, shift=beta-mean*scale; saves mean, invstd;
 * running_mean/var updated with `momentum` (unbiased var), num_batches_tracked (int64) += 1.
 * eval (training==0): scale/shift from the running statistics; stats may be NULL. */
int mpgan_bn_finalize(const double* stats, int64_t pixels, int32_t c, const float* gamma, const float* beta,
                      float eps, float momentum, int training, float* running_mean, float* running_var,
                      int64_t* num_batches_tracked, float* mean, float* invstd, float* scale, float* shift,
                      void* stream);
/* y = act(x*scale[c] + shift[c]) (+ res).  act: NONE, PRELU (slope read from *alpha), LEAKY (slope = *alpha
 * when alpha != NULL else 0.2), TANH.  scale/shift may be NULL (identity).  res may be NULL. */
int mpgan_bn_act_apply(int dtype, const void* x, int64_t ldx, int64_t pixels, int32_t c, const float* scale,
                       const float* shift, int act, const float* alpha, float leaky_slope, const void* res,
                       int64_t ldres, void* y, int64_t ldy, void* stream);
/* training-mode finalize + apply in one launch: every thread derives scale/shift of its own channels from the fp64
 * statistics (the arithmetic of mpgan_bn_finalize); the first block also writes mean/invstd/scale/shift (saved for
 * the backward pass) and updates running_mean/var and num_batches_tracked. */
int mpgan_bn_train_apply(int dtype, const void* x, int64_t ldx, int64_t pixels, int32_t c, const double* stats,
                         const float* gamma, const float* beta, float eps, float momentum, float* running_mean,
                         float* running_var, int64_t* num_batches_tracked, float* mean, float* invstd, float* scale,
                         float* shift, int act, const float* alpha, float leaky_slope, const void* res,
                         int64_t ldres, void* y, int64_t ldy, void* stream);
/* backward of y = act(bn(x)): pass 1 reduces  sums[0:C]=sum g, sums[C:2C]=sum g*xhat, sums[2C]=sum dy*min(z,0)
 * (PReLU slope grad), all fp64 accumulating;  pass 2 writes dx and accumulates dgamma/dbeta/dalpha (fp32) and, when
 * dbias != NULL, the bias gradient of the convolution that produced x: dbias[c] += sum_p dx[p,c]. */
int mpgan_bn_act_bwd_reduce(int dtype, const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t pixels,
                            int32_t c, const float* mean, const float* invstd, const float* scale,
                            const float* shift, int act, const float* alpha, float leaky_slope, double* sums,
                            void* stream);
int mpgan_bn_act_bwd_apply(int dtype, const void* dy, int64_t lddy, const void* x, int64_t ldx, int64_t pixels,
                           int32_t c, const float* mean, const float* invstd, const float* scale,
                           const float* shift, int act, const float* alpha, float leaky_slope, const double* sums,
                           float* dgamma, float* dbeta, float* dalpha, float* dbias, void* dx, int64_t lddx,
                           void* stream);

/* ---- elementwise helpers on channels-last tensors ---- */
/* y[p, 0:c] = a[p, 0:c] (+ b[p, 0:c]) with independent pixel strides (residual add, concat copy, casts). */
int mpgan_add_copy(int dtype_in, const void* a, int64_t lda, const void* b, int64_t ldb, int dtype_out, void* y,
                   int64_t ldy, int64_t pixels, int32_t c, void* stream);
/* nn.Tanh (GAN_final.py:117) forward and backward on a flat tensor: y = tanh(x);  dx = dy*(1-y^2). */
int mpgan_tanh_fwd(int dtype_in, const void* x, int dtype_out, void* y, int64_t n, void* stream);
int mpgan_tanh_bwd(int dtype, const void* dy, const void* y, void* dx, int64_t n, void* stream);
/* per-channel column sum: out[c] += sum_p x[p,c]  (conv bias gradient). fp32 accumulate into out. */
int mpgan_colsum(int dtype, const void* x, int64_t ldx, int64_t pixels, int32_t c, float* out, void* stream);

/* ---- nn.Linear after Flatten (GAN_final.py:200-201; test_runs/GAN.py:176-181) ----
 * x: (batch, k) in `dtype` (channels-last flatten order), w: (j, k) in `dtype` pre-permuted to the same order,
 * bias fp32 (j) or NULL, y fp32 (batch, j).  fwd accumulates into y (caller zeroes y). */
int mpgan_linear_fwd(int dtype, const void* x, const void* w, const float* bias, float* y, int32_t batch,
                     int64_t k, int32_t j, void* stream);
/* dx (batch,k) `dtype` = dy (batch,j) fp32 * w;   dw (j,k) fp32 += dy^T x;  db (j) += sum dy.  NULL skips. */
int mpgan_linear_bwd(int dtype, const void* x, const void* w, const float* dy, void* dx, float* dw, float* db,
                     int32_t batch, int64_t k, int32_t j, void* stream);
/* (c, spatial) <-> (spatial, c) permutation of each row of a (rows, c*spatial) matrix, with dtype conversion:
 * to_cl=1: dst[r][s][c] = src[r][c][s];  to_cl=0: dst[r][c][s] (+)= src[r][s][c]. */
int mpgan_permute_flatten(int dtype_src, const void* src, int dtype_dst, void* dst, int32_t rows, int32_t c,
                          int64_t spatial, int to_cl, int accumulate, void* stream);

/* ---- losses ----
 * nn.Sigmoid (GAN_final.py:203) on the (n) fp32 logits and its backward dz = dprob * p * (1-p). */
int mpgan_sigmoid_fwd(const float* z, float* prob, int32_t n, void* stream);
int mpgan_sigmoid_bwd(const float* dprob, const float* prob, float* dz, int32_t n, void* stream);
/* F.binary_cross_entropy (GAN_final.py:244-245) on probabilities, torch's clamp semantics:
 * loss += weight * mean(-(t*max(log p,-100) + (1-t)*max(log1p(-p),-100)));  loss (1) fp32 accumulates.
 * backward: dprob = gscale * weight/n * (p - t)/max(p(1-p), 1e-12)   (gscale: device scalar or NULL = 1). */
int mpgan_bce_fwd(const float* prob, const float* target, float weight, float* loss, int32_t n, void* stream);
int mpgan_bce_bwd(const float* prob, const float* target, float weight, const float* gscale, float* dprob,
                  int32_t n, void* stream);
/* F.l1_loss (GAN_final.py:247-248): loss += weight * mean|a-b| ;  da = gscale*weight/n * sign(a-b) */
int mpgan_l1_fwd(int dtype, const void* a, const void* b, int64_t n, float weight, float* loss, void* stream);
int mpgan_l1_bwd(int dtype, const void* a, const void* b, int64_t n, float weight, const float* gscale, void* da,
                 int accumulate, void* stream);
/* one pass: *loss (fp32) and / or *loss64 (fp64) += weight * mean|a - b| (either may be NULL) and
 * da (+)= gscale * weight / n * sign(a - b) (da may be NULL; accumulate != 0 adds onto da's contents) -- F.l1_loss forward +
 * backward fused; the feature-matching loss of test_runs/GAN.py:288-298 accumulates its gradients straight into the
 * discriminator's backward tensors with it and sums its 16 terms in the fp64 slot. */
int mpgan_l1_fwd_bwd(int dtype, const void* a, const void* b, int64_t n, float weight, const float* gscale, float* loss,
                     double* loss64, void* da, int accumulate, void* stream);

/* ---- torch.optim.Adam (GAN_final.py:298-308), one launch over a flat fp32 buffer ----
 * state: 3 device floats {step count (int bits), step_size, sqrt(1-beta2^t)}; zero-initialised by the caller.
 * The call increments the device-side step count first (so a captured CUDA graph advances it on replay), then
 * applies exp_avg/exp_avg_sq/param updates with torch's formula.  Optionally writes a bf16 shadow copy. */
int mpgan_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                    float beta1, float beta2, float eps, float* state, void* bf16_shadow, void* stream);
/* dst = cast(src) for flat buffers (f32 <-> bf16). */
int mpgan_cast(int dtype_src, const void* src, int dtype_dst, void* dst, int64_t n, void* stream);
/* OTI [cy][taps][cx] -> transposed shadow [cx][taps][cy] with dtype conversion. */
int mpgan_weight_transpose(int dtype_src, const void* src, int dtype_dst, void* dst, int32_t cy, int32_t taps,
                           int32_t cx, void* stream);
/* the same for n bf16 tensors in one launch: table = n x 5 device int64 {src, dst, cy, taps, cx}; max_elems = the largest
 * cy*taps*cx (grid sizing) */
int mpgan_weight_transpose_batch(const int64_t* table_dev, int32_t n, int32_t max_elems, void* stream);

/* ---- RandSpatialCropSamplesd gather (test_runs/GAN.py:263-272,313-337), bit-exact copy ----
 * vol: (batch, *S, c) channels-last; origins: device int32 (batch*num_samples, rank) in (D,H,W) order;
 * out: (batch*num_samples, roi.., c).  scatter_add is its deterministic backward (dvol += patches). */
int mpgan_patch_gather(int dtype, const void* vol, int32_t batch, int32_t rank, const int32_t* spatial, int32_t c,
                       const int32_t* origins, int32_t num_samples, int32_t roi, void* out, void* stream);
int mpgan_patch_scatter_add(int dtype, const void* dpatch, int32_t batch, int32_t rank, const int32_t* spatial,
                            int32_t c, const int32_t* origins, int32_t num_samples, int32_t roi, void* dvol,
                            void* stream);

/* ---- fused tail of a generator UNet (MONAI UNet top level: ConvT(..->1) -> BatchNorm(1) -> PReLU -> ResidualUnit(1->1,
 * conv only), call site GAN_final.py:106-114) on a one-channel (n, h, w) bf16 image, training mode:
 *   hmap = prelu(batchnorm(c));  y = conv3x3(hmap, w9, pad 1) + bias + hmap
 * stats: the fp64 {sum, sum of squares} of c; running statistics / saved mean, invstd, scale, shift are updated as by
 * mpgan_bn_train_apply.  h_out may be NULL (no backward pass will follow).  stats == NULL: evaluation mode -- scale /
 * shift are INPUTS (mpgan_bn_finalize of the running statistics) and no statistic is written. */
int mpgan_c1_tail_fwd(const void* c_bf16, int32_t n, int32_t h, int32_t w, const double* stats, const float* gamma,
                      const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                      int64_t* num_batches_tracked, float* mean, float* invstd, float* scale, float* shift,
                      const float* alpha, const void* w9_bf16, const float* bias, void* h_out_bf16, void* y_out_bf16,
                      void* stream);
/* backward twin: dh = conv3x3^T(dy, w9) + dy (bf16, same layout) and the BatchNorm(1) + PReLU backward reduction of c in
 * the same pass: sums3[0] += sum dz, sums3[1] += sum dz*xhat, sums3[2] += sum_{z<=0} dh*z (the layout
 * mpgan_bn_act_bwd_apply reads with c == 1); mean / invstd / scale / shift = the values saved by the forward. */
int mpgan_c1_tail_bwd_reduce(const void* dy_bf16, const void* c_bf16, int32_t n, int32_t h, int32_t w, const float* mean,
                             const float* invstd, const float* scale, const float* shift, const float* alpha,
                             const void* w9_bf16, void* dh_bf16, double* sums3, void* stream);

/* ---- one-input-channel 3x3 weight gradient through the tensor cores (conv_c1col.cu) ----
 * im2col_c1: x (n, ih, iw) contiguous bf16, one channel -> xcol (n, oh, ow, 16) bf16: the 9 taps of every output pixel
 *   (zero padded borders) followed by 7 zeros.  The weight gradient is then mpgan_tc_conv_wgrad of the 1x1 layer
 *   xcol(16) -> dY(cy) into a zeroed fp32 dw16[cy][16], and fold_dw16 adds dw16[c][t<9] into dw[c][9]. */
int mpgan_im2col_c1(const void* x_bf16, int32_t n, int32_t ih, int32_t iw, int32_t oh, int32_t ow, int32_t stride,
                    int32_t pad, void* xcol_bf16, void* stream);
int mpgan_fold_dw16(const float* dw16, int32_t cy, float* dw, void* stream);

/* ---- one-channel layers of the rank-3 networks (conv_c1vol.cu; the reference's literal volumes: GAN_final.py:107
 * dimensions=3, :167-169 Conv3d(1, 64, 3), MONAI UNet's 1 -> 16 entry convolutions / 32 -> 1 ConvTranspose / 1 -> 1 tail) ----
 * A 3x3x3 convolution with one input channel == a 1x1x1 convolution over xcol (n, *ys, 32) = the 27 taps of every output
 * voxel + 5 zeros, which the rank-3 tcgen05 kernels run (mpgan_tc_conv_fprop / _wgrad with cx = 32):
 * im2col_c1_vol: x (n, *xs3) one channel contiguous bf16 -> xcol (n, *ys3, 32) bf16 (zero padded borders).
 * col2im_c1_vol: t (n, *ys3, 32) bf16 = per-tap partial products of a data gradient / ConvTranspose (the 1x1x1 convolution
 *   of the Y-grid tensor with the [32][cy] transposed weights) -> x (n, *xs3) one channel bf16:
 *   x[q] = bias + res[q] + sum over taps r with (q + pad - r) % stride == 0 of t[(q + pad - r) / stride][r].
 * fold_dw32: dw[c][27] += dw32[c][32] (first 27 columns of the 1x1x1 weight gradient).
 * stencil27 / stencil27_wgrad: the 1 -> 1 channel k3 s1 p1 layer as direct 27-point stencils (dtype MPGAN_F32 / MPGAN_BF16;
 *   direction 0: y = bias + conv(x, w27); 1: dx = conv^T(dy, w27) + res; wgrad: dw27[t] += sum dy * x(shifted), dbias += sum dy). */
int mpgan_im2col_c1_vol(const void* x_bf16, int32_t n, const int32_t* xs3, const int32_t* ys3, int32_t stride, int32_t pad,
                        void* xcol_bf16, void* stream);
int mpgan_col2im_c1_vol(const void* t_bf16, int32_t n, const int32_t* xs3, const int32_t* ys3, int32_t stride, int32_t pad,
                        const float* bias, const void* res_bf16, void* x_bf16, void* stream);
int mpgan_fold_dw32(const float* dw32, int32_t cy, float* dw, void* stream);
int mpgan_stencil27(int dtype, int direction, const void* in, int32_t n, int32_t d, int32_t h, int32_t w, const void* w27,
                    const float* bias, const void* res, void* out, void* stream);
int mpgan_stencil27_wgrad(int dtype, const void* x, const void* dy, int32_t n, int32_t d, int32_t h, int32_t w, float* dw27,
                          float* dbias, void* stream);

/* ---- intensity transforms / volume metrics around the generator (SURVEY.md section 8f, N1 / N2 / N5) ----
 * MONAI ScaleIntensityRangePercentilesd (reference: GAN_final.py:386-394 lower=1 upper=99 -> [-1,1];
 * inferrence.py:152-160,190-198 lower=0 upper=100 -> [0,255] followed by np.round), torchmetrics
 * MeanAbsoluteError / MeanSquaredError (inferrence.py:170-176, metrics.py:213-218), scikit-image SSIM / PSNR
 * (psnr_ssim_metric.py:88-95; PSNR is host arithmetic over err_sums) and mutual information (the score of
 * the reference's code/eval XML files, restated as scikit-image's normalized_mutual_information).
 * order_stats: out[r] = the ranks[r]-th smallest value (0-based, exact) of the fp32 volume x[0..n); ranks is a DEVICE
 *   array of nranks <= 4 int64; workspace of mpgan_order_stats_workspace(nranks) bytes (caller-owned, overwritten).
 * minmax: the same contract restricted to ranks in {0, n-1} (the 0 / 100 percentiles): one min/max reduction pass.
 * rescale_intensity: y = ((x - a_min) / (a_max - a_min)) * (b_max - b_min) + b_min  (x - a_min + b_min when
 *   a_max == a_min), each step rounded to fp32; optional clip to [clip_lo, clip_hi]; optional round-half-even;
 *   out_dtype 0 = fp32, 2 = fp16.
 * err_sums: out2[0] += sum |a-b|, out2[1] += sum (a-b)^2  (device fp64, zero-initialised by the caller). */
size_t mpgan_order_stats_workspace(int32_t nranks);
int mpgan_order_stats(const float* x, int64_t n, const int64_t* ranks, int32_t nranks, float* out, void* workspace,
                      size_t workspace_bytes, void* stream);
int mpgan_minmax(const float* x, int64_t n, const int64_t* ranks, int32_t nranks, float* out, void* workspace,
                 size_t workspace_bytes, void* stream);
int mpgan_rescale_intensity(const float* x, int64_t n, float a_min, float a_max, float b_min, float b_max, int clip,
                            float clip_lo, float clip_hi, int round_half_even, int out_dtype, void* y, void* stream);
int mpgan_err_sums(const float* a, const float* b, int64_t n, double* out2, void* stream);
/* ssim_sums: scikit-image structural_similarity (psnr_ssim_metric.py:88-95) without its final mean:
 *   out[i] += sum over the interior voxels (window inside the image) of item i of the SSIM map
 *   S = (2 ux uy + c1)(2 vxy + c2) / ((ux^2 + uy^2 + c1)(vx + vy + c2)),  v* = cov_norm (u** - u* u*),
 *   ux, uy, uxx, uyy, uxy = x, y, x*x, y*y, x*y filtered by the separable window `taps` (fp64 accumulation).
 *   a, b: items x (d, h, w) contiguous fp32; rank 2 = d == 1 with no filtering along d.  taps: HOST array of win
 *   fp64 weights (uniform or Gaussian), read at call time; win odd, 3..15, <= every filtered extent.  out: device fp64
 *   [items], zero-initialised by the caller; mssim = out[i] / (interior voxel count). */
int mpgan_ssim_sums(const float* a, const float* b, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                    const double* taps, int32_t win, double c1, double c2, double cov_norm, double* out, void* stream);
/* mutual_info: the numpy/scipy computation of scikit-image's normalized_mutual_information(x, y, bins), and plain mutual
 * information from the same joint histogram, for `items` pairs x = a[i*n .. (i+1)*n), y = b[...] (contiguous fp32):
 *   range   lo = min, hi = max of each image separately; lo == hi: lo = fl(lo - 0.5), hi = fl(hi + 0.5) (fp32).
 *   edges   np.histogramdd's fp32 edges, every step rounded to fp32 (no FMA): delta = hi - lo, step = delta / bins;
 *           e_i = i step + lo for 0 <= i < bins, or (i / bins) delta + lo when step underflows to 0; e_bins = hi.
 *   bin     of v: searchsorted(e, v, side="right") - 1 in fp32 comparisons; v == e_bins goes into bin bins - 1.
 *           The table is non-decreasing unless step is subnormal (an image whose whole range is below ~1e-36), where
 *           numpy's own bins depend on the order of the values; the bin is then the kernel's walk over the table.
 *   counts  [i][r][c] = the voxels whose x falls in bin r and whose y falls in bin c (exact integers).
 *   out5    [i] = {H1, H2, H12, MI = H1 + H2 - H12, NMI = (H1 + H2) / H12} in nats, fp64, H(p) = -sum p log p with
 *           p = count / n and 0 log 0 = 0; H1 from the row sums, H2 from the column sums.  NMI is NaN when H12 == 0.
 *   Where numpy raises (a min or max that is NaN or +-inf), the item instead gets NaN in out5, NaN edges and all-zero
 *   counts; the other items are unaffected.
 * counts: device int64 [items][bins][bins]; edges: device fp32 [items][2][bins + 1] (x's then y's) or NULL; out5: device
 * fp64 [items][5]; all three are overwritten.  2 <= bins <= 128, 1 <= n <= 2^31 - 1.  workspace: device, at least
 * mpgan_mutual_info_workspace(items) bytes, overwritten. */
size_t mpgan_mutual_info_workspace(int32_t items);
int mpgan_mutual_info(const float* a, const float* b, int32_t items, int64_t n, int32_t bins, int64_t* counts,
                      float* edges, double* out5, void* workspace, size_t workspace_bytes, void* stream);

/* ---- foreground-masked metrics and Otsu's foreground mask ----
 * mask: device uint8, laid out like the images (items x n); a non-zero byte puts the voxel in the mask.  Voxels outside
 * the mask are never used, even when they hold NaN or +-inf (a select, not a multiply by 0).  An empty mask gives zero
 * counts, NaN scores and NaN edges, without any host synchronisation.
 * err_sums_masked: out3[0] += sum_m |a-b|, out3[1] += sum_m (a-b)^2, out3[2] += sum m (the voxels in the mask): err_sums
 *   restricted to the mask, in one pass.  out3: device fp64 [3], zero-initialised by the caller.
 * ssim_sums_masked: ssim_sums, but out[i] sums S only over the interior voxels whose CENTRE is in the mask, and
 *   count[i] += the number of those voxels (device fp64 [items], zero-initialised); the masked mean SSIM is
 *   out[i] / count[i].  The windows still read the unmasked neighbours, so S itself is unchanged.
 * mutual_info_masked: mutual_info of x[m], y[m]: lo / hi from the voxels in the item's mask only; edges, bins and
 *   entropies as mutual_info with p = count / (the voxels in the mask).  Same workspace. */
int mpgan_err_sums_masked(const float* a, const float* b, const uint8_t* mask, int64_t n, double* out3, void* stream);
int mpgan_ssim_sums_masked(const float* a, const float* b, const uint8_t* mask, int32_t rank, int32_t items, int32_t d,
                           int32_t h, int32_t w, const double* taps, int32_t win, double c1, double c2, double cov_norm,
                           double* out, double* count, void* stream);
int mpgan_mutual_info_masked(const float* a, const float* b, const uint8_t* mask, int32_t items, int64_t n, int32_t bins,
                             int64_t* counts, float* edges, double* out5, void* workspace, size_t workspace_bytes,
                             void* stream);
/* otsu_threshold: thr[i] = Otsu's threshold of x[i*n .. (i+1)*n) (fp32), scikit-image's threshold_otsu(image, nbins)
 * algorithm restated with this precision (scikit-image's versions differ in it, so no parity with one is claimed):
 *   1. lo, hi = min, max of the item.  Either non-finite: thr = NaN.  lo == hi: thr = lo.
 *   2. the bins + 1 fp32 edges of mutual_info (np.histogram(x, bins)'s), the counts of np.histogram (searchsorted bins,
 *      last bin closed) in int64.
 *   3. centres c_i = fl32(fl32(e_i + e_{i+1}) / 2).
 *   4. w1 = cumsum(counts), w2 = reverse cumsum(counts) (int64); mean1_i = (sum_{j<=i} fl64(counts_j c_j)) / w1_i and
 *      mean2_i = (sum_{j>=i} fl64(counts_j c_j)) / w2_i, each sum sequential in fp64 (mean2's from the top);
 *      var_i = fp64(w1_i w2_{i+1}) (d d), d = mean1_i - mean2_{i+1}, the product w1_i w2_{i+1} in int64, i < bins - 1;
 *      every operation rounded, no FMA.
 *   5. idx = the first index of the maximum of var (np.argmax: the first NaN, an empty lower class, wins); thr = c_idx.
 *   2 <= bins <= 256, 1 <= n <= 2^31 - 1.  thr: device fp32 [items], overwritten.  workspace: device, at least
 *   mpgan_otsu_threshold_workspace(items, bins) bytes, overwritten.
 * threshold_mask: mask[i*n + j] = x[i*n + j] > thr[i] ? 1 : 0 (so a NaN threshold gives an empty mask); thr: device fp32
 *   [items]; mask: device uint8 [items * n], overwritten. */
size_t mpgan_otsu_threshold_workspace(int32_t items, int32_t bins);
int mpgan_otsu_threshold(const float* x, int32_t items, int64_t n, int32_t bins, float* thr, void* workspace,
                         size_t workspace_bytes, void* stream);
int mpgan_threshold_mask(const float* x, const float* thr, int32_t items, int64_t n, uint8_t* mask, void* stream);

/* ---- connected components and binary morphology of masks (scipy.ndimage; MONAI's KeepLargestConnectedComponent and
 * FillHoles steps), to clean the Otsu mask into a head mask ----
 * Images: `items` uint8 masks of (d, h, w) contiguous voxels, item-major, non-zero = "in"; rank 3 images are (d, h, w),
 *   rank 2 images (h, w) with d == 1 (at rank 3 a d == 1 image has every voxel on a face).  1 <= d h w <= 2^31 - 1.
 * Structure: scipy.ndimage.generate_binary_structure(rank, connectivity), 1 <= connectivity <= rank: the neighbours at
 *   offsets in {-1, 0, 1}^rank with |o|_1 <= connectivity (4 / 8 at rank 2, 6 / 18 / 26 at rank 3).
 * label: scipy.ndimage.label(mask, structure): labels[v] = 0 in the background, else 1 .. k numbering the components in
 *   raster order of their smallest linear index; count[i] = k of item i (device int32 [items], so no synchronisation).
 * largest_component: out = the "in" voxels of the component with the most voxels, ties to the lowest label
 *   (np.argmax(np.bincount(labels)[1:])); an empty image stays empty.
 * fill_holes: scipy.ndimage.binary_fill_holes(mask, structure): mask | every background component (under the same
 *   structure) that touches no face of the image.
 * binary_morphology: scipy.ndimage.binary_erosion (op 0) / binary_dilation (op 1) with the structure, border_value 0
 *   (erosion removes "in" voxels whose structure reaches outside the image) and iterations >= 1.
 * Outputs (labels int32, out uint8 0 / 1, item-major like the mask) are overwritten and must not overlap the mask.
 * workspace: device, at least mpgan_morphology_workspace(items, d, h, w) bytes (about 8 bytes per voxel: parents and
 * sizes; ~0.5 GB for one 256 x 512 x 512 image), overwritten.  Labelling has a fixed launch count (block union-find), so
 * every call can be captured in a CUDA graph; the result does not depend on the order of the atomics. */
size_t mpgan_morphology_workspace(int32_t items, int32_t d, int32_t h, int32_t w);
int mpgan_label(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w, int32_t connectivity,
                int32_t* labels, int32_t* count, void* workspace, size_t workspace_bytes, void* stream);
int mpgan_largest_component(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                            int32_t connectivity, uint8_t* out, void* workspace, size_t workspace_bytes, void* stream);
int mpgan_fill_holes(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                     int32_t connectivity, uint8_t* out, void* workspace, size_t workspace_bytes, void* stream);
int mpgan_binary_morphology(const uint8_t* mask, int32_t rank, int32_t items, int32_t d, int32_t h, int32_t w,
                            int32_t connectivity, int32_t op, int32_t iterations, uint8_t* out, void* workspace,
                            size_t workspace_bytes, void* stream);

/* ---- sliding-window inference (MONAI 0.4.0 sliding_window_inference, the call minipig_inference.py:110-114 leaves
 * commented out; constant padding only) ----
 * Geometry table: int32 words, built once per call by the caller, passed twice: `geom` (HOST copy, validated in full
 * before any launch) and `geom_dev` (a DEVICE copy of the same words, 8-byte aligned, read by the kernels);
 * geom_words = its length.  Spatial dims are (D, H, W); rank 2 uses a trivial D (size 1, roi 1, lo 0, one window
 * starting at 0, coverage [0, 0], tap 1).  With P_d = max(S_d, roi_d) the padded extent:
 *   [0, 16)   header: rank, S[3], roi[3], lo[3], n[3], 0, 0, 0   (lo_d = max(roi_d - S_d, 0) / 2; n_d windows along d)
 *   starts    n[0] + n[1] + n[2] words: window starts per dim in padded coordinates, increasing, s + roi_d <= P_d
 *   cover     2 (P[0] + P[1] + P[2]) words: per dim and padded coordinate p, {j_first, j_last}, the windows covering p
 *             (only the coordinates of the unpadded image are read and validated)
 *   taps      at the next even word: roi[0] + roi[1] + roi[2] fp64 importance taps per dim, in (0, 1]
 * Windows are the Cartesian product of the per-dim starts, first dim slowest, image-major: window k of the global order
 * is image k / nwin, nwin = n[0] n[1] n[2].
 * window_gather: out (count, channels, *roi) = windows [first, first + count) of x (batch, channels, *S), cval outside S
 *   (an exact copy).
 * window_blend: pred (batch * nwin, channels, *roi) -> out (batch, channels, *S):
 *   out(p) = sum_k w(p - s_k) pred_k(p - s_k) / sum_k w(p - s_k) over the windows covering p, w = prod_d taps_d,
 *   fp64 sums in window order, one rounding to fp32; gather-style (no atomics), bit-identical run to run. */
int mpgan_window_gather(const float* x, int32_t batch, int32_t channels, const int32_t* geom, const int32_t* geom_dev,
                        int64_t geom_words, int64_t first, int64_t count, float cval, float* out, void* stream);
int mpgan_window_blend(const float* pred, int32_t batch, int32_t channels, const int32_t* geom, const int32_t* geom_dev,
                       int64_t geom_words, float* out, void* stream);

/* ---- linear resampling between physical grids (ITK 5.1 ResampleImageFilter + IdentityTransform +
 * LinearInterpolateImageFunction on float pixels: ResampleT1T2d, code/GAN/transforms.py:79-213, the first step of
 * GAN_final.py:381-398 and inferrence.py:119-139) ----
 * in: items x (in_z, in_y, in_x) contiguous fp32; out: items x (out_z, out_y, out_x), every item on one geometry.
 * in_size / out_size: HOST int32[3] in ITK axis order (x, y, z), each in [1, 2^22]; rank 2 has z extents 1.
 * map: HOST fp64[24] = o_out[3], M_out[9] row-major, o_in[3], N_in[9] row-major, with M_out = D_out diag(S_out) and
 *   N_in = inverse(D_in diag(S_in)); all finite; rank 2: z row and column of M_out and N_in those of the identity, z
 *   origins 0.  Sizes and map are read during the call and passed to the kernel by value.
 * Per output voxel i = (i_x, i_y, i_z), in fp64 with every operation rounded (no FMA), in this order:
 *   p_k = ((o_out_k + M_out[k,0] i_x) + M_out[k,1] i_y) + M_out[k,2] i_z
 *   c_k = ((N_in[k,0] (p_0 - o_in_0)) + N_in[k,1] (p_1 - o_in_1)) + N_in[k,2] (p_2 - o_in_2)
 *   outside unless -0.5 <= c_k < n_k - 0.5 for every k: out = default_value;
 *   else per axis b = max(floor(c), 0), d = c - b (d <= 0 -> 0), upper neighbour min(b + 1, n - 1), not read at d = 0;
 *   lerps a + (b - a) d along x, then y, then z (ITK's EvaluateOptimized nesting), rounded once to fp32. */
int mpgan_resample_linear(const float* in, int64_t items, int32_t rank, const int32_t in_size[3],
                          const int32_t out_size[3], const double map[24], float default_value, float* out,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPGAN_H_ */
