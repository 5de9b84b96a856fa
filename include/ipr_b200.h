/*
 * ipr_b200.h -- C ABI of libipr_b200.so: hand-written sm_100a CUDA kernels for the IPR-GAN hot path.
 *
 * The reference (dingsheng-ong/ipr-gan) is pure Python and has no FFI of its own; its "plugin"
 * surface is the Python API of tools/*.py, models/wrappers.py and networks/*.py.  Each entry point
 * below replaces the PyTorch op sequence of one reference function (cited file:line, paths relative
 * to the reference root) and is what a ctypes binding inside that function would call
 * (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - tensors are contiguous, NCHW, fp32 unless stated;
 *   - the caller owns every buffer including workspaces; the library never allocates or frees
 *     device memory and keeps no pointer after the call returns;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never synchronises,
 *     never touches the default stream, and is CUDA-graph capturable;
 *   - return value: 0 = OK; < 0 = argument error found on the host before any launch
 *     (IPR_E_*); > 0 = cudaError_t reported by the launch.  ipr_strerror() names both.
 *   - there is no CPU fallback.
 */
#ifndef IPR_B200_H
#define IPR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IPR_OK              0
#define IPR_E_NULL         -1   /* a required pointer is NULL                       */
#define IPR_E_SHAPE        -2   /* inconsistent / non-positive dimensions           */
#define IPR_E_UNSUPPORTED  -3   /* valid but outside what the kernels cover         */
#define IPR_E_ALIGN        -4   /* pointer alignment requirement violated           */
#define IPR_E_WORKSPACE    -5   /* workspace too small                              */

typedef void *ipr_stream_t;     /* cudaStream_t */

int         ipr_version(void);
const char *ipr_strerror(int code);
/* number of kernels this library has launched in this process (for bench.py's gpu_launches) */
uint64_t    ipr_launch_count(void);

/* ------------------------------------------------------------------ black-box trigger path */

/* y = x; y[win] = y[win]*bg + (1-bg)*fg  with win = rows [row0,row0+s) x cols [col0,col0+s).
 * Replaces PasteWatermark.forward (tools/paste_watermark.py:45-52) and
 * RandomNoisePatch.forward (tools/random_noise_patch.py:38-45).  fg: (C,s,s), bg: (s,s).
 * Bit-exact: two rounded ops (mul, then mul+add without FMA), as the reference's two in-place ops. */
int ipr_paste_patch_f32(const float *x, float *y, const float *fg, const float *bg,
                        int64_t batch, int channels, int height, int width,
                        int size, int row0, int col0, ipr_stream_t stream);

/* Fused trigger build for one training step: ywm = paste(x) as above AND xwm = transform_dist(z)
 * in ONE launch (models/wrappers.py:49-51 with the DCGAN config's fn_inp/fn_out). */
int ipr_trigger_pair_f32(const float *x, float *ywm, const float *fg, const float *bg,
                         int64_t batch, int channels, int height, int width, int size, int row0, int col0,
                         const float *z, float *xwm, int64_t z_numel, ipr_stream_t stream);

/* out = 1*bg + (1-bg)*x[win]  -> (batch, C, s, s).
 * Replaces PasteWatermark.apply_mask / RandomNoisePatch.apply_mask
 * (tools/paste_watermark.py:54-61, tools/random_noise_patch.py:47-54). */
int ipr_crop_patch_f32(const float *x, float *out, const float *bg,
                       int64_t batch, int channels, int height, int width,
                       int size, int row0, int col0, ipr_stream_t stream);

/* The same crop followed by the evaluation loop's post-processing, out = (clamp(crop, -1, 1) + 1) / 2 -- one pass
 * instead of crop + clamp + add + div (experiments/image_generation.py:141-149, 208-209; sign_flip.py:59-75). */
int ipr_crop_postproc_f32(const float *x, float *out, const float *bg,
                          int64_t batch, int channels, int height, int width,
                          int size, int row0, int col0, ipr_stream_t stream);

/* The same crop followed by out = clamp(crop, 0, 1): the post-processing of normalized=False outputs, which are already
 * in data range 1 (the SRGAN family), before the per-sample SSIM and pHash of the verification loop
 * (experiments/image_super_resolution.py:229).  Replaces apply_mask + clamp_(0, 1); NaN propagates and -0 stays -0
 * as in torch.clamp.  Same arguments and error codes as ipr_crop_postproc_f32. */
int ipr_crop_clamp01_f32(const float *x, float *out, const float *bg,
                         int64_t batch, int channels, int height, int width,
                         int size, int row0, int col0, ipr_stream_t stream);

/* out = z; out[:, mask[j]] = constant.  Replaces RandomBitMask.forward (tools/random_bitmask.py:12-15).
 * mask: n int64 indices in [0, z_dim). */
int ipr_bitmask_scatter_f32(const float *z, float *out, const int64_t *mask,
                            int64_t batch, int z_dim, int n, float constant, ipr_stream_t stream);

/* out = 0.5*(1+erf(z/sqrt(2)))*sqrt(2*pi).  Replaces TransformDist.forward (tools/transform_dist.py:9-11). */
int ipr_transform_dist_f32(const float *z, float *out, int64_t numel, ipr_stream_t stream);

/* out = z*(1-a) + a*w with a, w of length dim broadcast over the batch.
 * Replaces TransformVar.forward (tools/transform_var.py:12-13). */
int ipr_transform_var_f32(const float *z, float *out, const float *a, const float *w,
                          int64_t batch, int dim, ipr_stream_t stream);

/* ------------------------------------------------------------------ watermark reconstruction loss (SSIM) */

/* Workspace (bytes) for ipr_ssim_fwd_bwd_f32 / ipr_ssim_per_sample_f32 on this shape. */
size_t ipr_ssim_workspace_bytes(int64_t batch, int channels, int height, int width);

/* loss = 1 - mean_{n,c} mean_{valid map} SSIM(x', y'),   x' = normalized ? (x+1)/2 : x  (same for y)
 * dx   = grad_scale * d loss / d x            (y is a constant, models/wrappers.py:49-51)
 * One pass over HBM: reads x and y once, writes dx once; the scalar loss is produced by a second,
 * single-CTA launch that adds the per-CTA partial sums in a fixed order (deterministic).
 * Replaces Loss.__call__ + ssim() (tools/loss.py:10-20, 82-85) -> pytorch_msssim.SSIM(data_range=1)
 * forward AND its autograd backward.  11-tap sigma-1.5 valid separable window; H, W >= 11.
 * dx may be NULL (forward only).  The value stored is loss * loss_scale (1 for the plain loss; 1/world when the
 * scalar lands in a metrics slot that a summing data-parallel all-reduce turns into the global mean). */
int ipr_ssim_fwd_bwd_f32(const float *x, const float *y, float *dx, float *loss,
                         void *workspace, size_t workspace_bytes,
                         int64_t batch, int channels, int height, int width,
                         int normalized, float grad_scale, float loss_scale, ipr_stream_t stream);

/* out[n] = mean_{c, valid map} SSIM(x[n], y[n])  (data_range 1, no de-normalisation).
 * Replaces pytorch_msssim.ssim(wm_x, wm_y, data_range=1, size_average=False)
 * (experiments/image_generation.py:211). */
int ipr_ssim_per_sample_f32(const float *x, const float *y, float *out,
                            void *workspace, size_t workspace_bytes,
                            int64_t batch, int channels, int height, int width, ipr_stream_t stream);

/* ------------------------------------------------------------------ white-box signature */

#define IPR_SIGN_MAX_LAYERS 64

typedef struct {
    const float *gamma;   /* normalisation-layer scale vector (device)               */
    const float *sign;    /* +1/-1 signature vector (device)                         */
    float       *grad;    /* d loss / d gamma destination (device) or NULL            */
    int32_t      n;       /* channels in this layer                                  */
    int32_t      reserved;
} ipr_sign_layer_t;

/* loss = sum_layers mean_c relu(gamma0 - gamma_c * sign_c);  grad_c = -grad_scale*sign_c/n_layer where active.
 * accumulate != 0 adds into grad instead of overwriting (fused-arena use).
 * `layers_host` is a HOST array of n_layers (<= IPR_SIGN_MAX_LAYERS) entries; it is copied into the
 * kernel parameters, so it may be freed right after the call.
 * grad pointers may be NULL (loss only: the gradient then rides in the BatchNorm backward, ipr_bn_relu_bwd_bf16);
 * the value stored is loss * loss_scale.
 * Replaces SignLossModel.forward (tools/sign_model.py:42-49) and its backward. */
int ipr_sign_loss_fwd_bwd_f32(const ipr_sign_layer_t *layers_host, int n_layers, float gamma0,
                              float grad_scale, int accumulate, float loss_scale, float *loss, ipr_stream_t stream);

/* counts[0] = #{c : sign(gamma_c) != sign_c} (gamma == 0 counts as wrong), counts[1] = total bits.
 * Replaces SignLossModel.compute_ber (tools/sign_model.py:51-60); integer, bit-exact. */
int ipr_sign_ber_i32(const ipr_sign_layer_t *layers_host, int n_layers, int32_t *counts,
                     ipr_stream_t stream);

/* ------------------------------------------------------------------ verification (pHash p-value) */

/* Bicubic up-sampling, align_corners=False, A=-0.75, border-replicated taps, with the operation
 * order of torch's CPU kernel (F.interpolate(..., mode='bicubic'), tools/phash_pvalue.py:28-29):
 * bit-exact against it (tests/test_gpu_ipr_ops.py::test_bicubic_bit_exact, tests/bicubic_ref.py).  x: (planes, hin, win) -> out: (planes, hout, wout). */
int ipr_bicubic_resize_f32(const float *x, float *out, int64_t planes,
                           int hin, int win, int hout, int wout, ipr_stream_t stream);

/* 16x64 DCT matrix used by the PDQ hash (host side, double cos -> float). */
void ipr_pdq_dct_matrix_host(float *d_host);

/* hash[n] = 256-bit PDQ hash (8 x uint32, bit k = word k/32, bit k%32; k = 16*i+j of the DCT block)
 * of image n after the reference's float->uint8 conversion (x*255 truncated, wrapped to 0..255).
 * img: (batch, 3, height, width) fp32; 8 <= height, width <= 64 (larger: IPR_E_UNSUPPORTED).
 * dct: device copy of ipr_pdq_dct_matrix_host().  coeffs (optional, may be NULL): (batch, 256) DCT block.
 * Replaces compute_hash (tools/phash_pvalue.py:7-17) -> pdqhash.compute. */
int ipr_pdq_hash_f32(const float *img, uint32_t *hash, float *coeffs, const float *dct,
                     int64_t batch, int height, int width, ipr_stream_t stream);

/* r[n] = 256 - popcount(hx[n] ^ hy[n]);  p[n] = ptable[r[n]]   (ptable: 257 fp32 entries
 * 1 - Binom(256, 1/2).cdf(r-1), built on the host exactly as tools/phash_pvalue.py:36 does).
 * Replaces tools/phash_pvalue.py:34-37. */
int ipr_hash_pvalue(const uint32_t *hx, const uint32_t *hy, const float *ptable,
                    float *p, int32_t *r, int64_t batch, ipr_stream_t stream);


/* ------------------------------------------------------------------ dense layers (tcgen05 implicit GEMM) */

#define IPR_TG_MAX_TAPS   16
#define IPR_TG_MAX_PHASES 4

/* epilogue modes */
#define IPR_EPI_LINEAR      0   /* out = acc / sigma                          -> bf16 NHWC (+ optional column stats) */
#define IPR_EPI_BIAS_LRELU  1   /* out = lrelu(acc / sigma + bias[n], slope)  -> bf16 NHWC                           */
#define IPR_EPI_MASK        2   /* out = acc / sigma * (mask[m,n] > 0 ? 1 : slope) -> bf16 NHWC (activation backward) */
#define IPR_EPI_TANH_NCHW   3   /* out = tanh(acc), columns < n_valid          -> fp32 NCHW                          */
#define IPR_EPI_LINEAR_F32  4   /* out = acc / sigma                          -> fp32 NHWC                           */
#define IPR_EPI_LINEAR_NCHW 5   /* out = acc / sigma, columns < n_valid        -> fp32 NCHW                          */

/* One "tap GEMM": for every phase p and output pixel m of a virtual grid (a_n x q_h x q_w)
 *     acc[m, n] = sum_{t < n_taps} sum_{c < a_c} A[img(m), s*qh(m) + dh[p][t], s*qw(m) + dw[p][t], c] * B[p][n][t*a_c + c]
 * with A an NHWC bf16 activation tensor read by TMA boxes (out-of-range pixels read as zero = padding) and B
 * packed bf16 weights.  s = 1 for a_parity == 0; for a_parity == 1 the tensor is addressed through its four
 * (row parity, column parity) sub-grids: tap_map[p][t] = 2*row_parity + col_parity and dh/dw are offsets in the
 * half-resolution grid (stride-2 convolution).  Output pixel of m: (qh*out_sh + out_oh[p], qw*out_sw + out_ow[p]).
 * This one kernel serves Conv2d k3s1 / k4s2 forward, ConvTranspose2d k4s2 (4 output-parity phases) and k3s1 forward,
 * their data gradients, and Linear (q_h = q_w = 1).
 * Replaces the cuDNN / cuBLAS calls under networks/conv_generator.py:8,13,21 and networks/sn_discriminator.py:9-21. */
typedef struct {
    const void *a;                 /* bf16 NHWC activations, 16-byte aligned                         */
    int32_t a_n, a_h, a_w, a_c;    /* a_c multiple of 64 (single-tap layers: multiple of 8, zero-extended) */
    int32_t a_parity;
    int32_t q_h, q_w;              /* virtual output grid per image; q_w*q_h divides or is divided by 128 */
    const void *b;                 /* bf16 [n_phases][n_total][n_taps*a_c]                           */
    int32_t n_total;               /* padded N (multiple of block_n)                                 */
    int32_t block_n;               /* 16, 32, 64, 128 or 256                                         */
    int32_t n_phases, n_taps;
    int8_t  tap_map[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t  tap_dh[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t  tap_dw[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int32_t epi_mode;
    float   slope;
    const float *sigma;            /* optional device scalar: acc is divided by it (spectral norm)   */
    const float *bias;             /* optional fp32 [n_total]                                        */
    const void  *mask;             /* IPR_EPI_MASK: bf16 tensor with the layout of `out`             */
    void   *out;
    int32_t out_h, out_w, out_c;   /* output tensor (a_n, out_h, out_w, out_c) NHWC (or NCHW fp32)   */
    int32_t out_sh, out_sw;
    int8_t  out_oh[IPR_TG_MAX_PHASES], out_ow[IPR_TG_MAX_PHASES];
    int32_t n_valid;               /* columns >= n_valid are not stored                              */
    float  *stats;                 /* optional [ipr_tapgemm_stats_rows()][2][n_total] partial column sums / sums of
                                      squares; their sum over rows is the statistic (IPR_EPI_MASK: sums only) */
    const float *scale;            /* optional fp32 [n_total], IPR_EPI_BIAS_LRELU only: out = lrelu(acc / sigma * scale[n] +
                                      bias[n]) -- an eval-mode BatchNorm (running statistics) folded into its layer */
} ipr_tapgemm_t;

/* number of M tiles of the launch described by d */
int ipr_tapgemm_m_tiles(const ipr_tapgemm_t *d_host);
/* rows the launch described by d writes into d->stats (every row is written; sum them) */
int ipr_tapgemm_stats_rows(const ipr_tapgemm_t *d_host);
int ipr_tapgemm_bf16(const ipr_tapgemm_t *d_host, ipr_stream_t stream);

/* Weight gradient of a tap-GEMM layer (tcgen05, MN-major operands, split-K over pixels):
 *     ws[split][p][n][t*x_c + c] = sum_{pixels m in the split} Y[pix_y(m)][n] * X[pix(m) + tap_t][c]
 * Y is the output-gradient-like operand (n = rows of dW), X the activation-like operand read with the
 * layer's taps.  y_parity / x_parity = 1: that tensor has twice the resolution of the (q_h, q_w) pixel
 * grid and is addressed through parity sub-grids (y_map[p] for Y; tap_map[p][t] for X).
 * Replaces the weight-gradient halves of cudnn convolution_backward / addmm backward under
 * networks/conv_generator.py and networks/sn_discriminator.py. */
typedef struct {
    const void *y; int32_t y_c, y_parity;
    const void *x; int32_t x_c, x_parity;
    int32_t n_imgs, q_h, q_w;
    int32_t n_phases, n_taps;
    int8_t  y_map[IPR_TG_MAX_PHASES];
    int8_t  tap_map[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t  tap_dh[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    int8_t  tap_dw[IPR_TG_MAX_PHASES][IPR_TG_MAX_TAPS];
    float  *workspace;             /* ipr_wgrad_workspace_bytes() */
    int32_t splits;
} ipr_wgrad_t;

size_t ipr_wgrad_workspace_bytes(const ipr_wgrad_t *d_host);
int    ipr_wgrad_total_kblocks(const ipr_wgrad_t *d_host);     /* 64-pixel blocks of the reduction */
int    ipr_wgrad_bf16(const ipr_wgrad_t *d_host, ipr_stream_t stream);

/* number of CTA tiles per split (the caller picks `splits` so that tiles*splits ~ number of SMs) */
int ipr_wgrad_tiles(const ipr_wgrad_t *d_host);

/* grad[row(n)*s_n + dst_off[p*k_total + k]] (+)= scale * sum_splits ws[split][p][n][k]   (dst_off < 0: skipped;
 * row(n) = row_map ? row_map[n] : n).  Adds the splits in a fixed order and scatters from the GEMM layout into the
 * parameter's own layout ((O,I,kh,kw), (I,O,kh,kw) or (O,I)). */
int ipr_wgrad_reduce_f32(const float *workspace, int splits, int phases, int n_rows, int k_total,
                         const int32_t *dst_off, const int32_t *row_map, int64_t s_n, float *grad,
                         int accumulate, float scale, ipr_stream_t stream);

/* The same reduction for plain Conv2d / ConvTranspose2d weights, destination-major (contiguous writes):
 *     grad[n*s_n + c*s_c + j] (+)= scale * sum_splits ws[split][p][n][t*x_c + c],   tap_of_host[j] = p*n_taps + t
 * for j < kk = phases*n_taps (<= 16).  Conv2d (O,I,kh,kw): s_n = I*kk, s_c = kk; ConvTranspose2d (I,O,kh,kw):
 * s_n = kk, s_c = O*kk.  tap_of_host is a HOST array (passed to the kernel by value). */
int ipr_wgrad_reduce_taps_f32(const float *workspace, int splits, int phases, int n_rows, int n_taps, int x_c,
                              const int32_t *tap_of_host, int kk, int64_t s_n, int64_t s_c, float *grad,
                              int accumulate, float scale, ipr_stream_t stream);

/* ------------------------------------------------------------------ memory-bound layers around the GEMMs */

/* out[(n,h,w)][k] (bf16, 32 columns = 64-byte rows) = x[n, c, h+kh-1, w+kw-1] for k = (kh*3+kw)*3 + c < 27, else 0;
 * x: (batch, 3, H, W) fp32 NCHW.  tanh_out (optional, same shape): x is multiplied by (1 - tanh_out^2)
 * (Tanh backward of networks/conv_generator.py:22 fused into the gather).  Feeds the first discriminator
 * convolution (networks/sn_discriminator.py:15, Cin = 3) and the last generator layer's gradients. */
int ipr_im2col3_bf16(const float *x, const float *tanh_out, void *out, int64_t batch, int height, int width,
                     ipr_stream_t stream);

/* Folds the nine taps of a 3-output-channel 3x3 layer: t = [batch*height*width][ld] fp32 (16-byte aligned,
 * ld >= 28 and a multiple of 4, batch < 65536) with column
 * (kh*3+kw)*3 + c holding tap (kh,kw) of channel c (produced by one plain GEMM over the 64-channel activation),
 * out[b][c][h][w] = act(sum_{kh,kw} t[(b, h+1-kh, w+1-kw)][(kh*3+kw)*3+c]), act = tanh if tanh_out else identity.
 * This is ConvTranspose2d(64,3,3,1,1)+Tanh of networks/conv_generator.py:21-22 and the input gradient of
 * Conv2d(3,64,3,1,1) of networks/sn_discriminator.py:15. */
int ipr_col2im3_f32(const float *t, float *out, int64_t batch, int height, int width, int ld, int tanh_out,
                    ipr_stream_t stream);

/* The same layer in ONE launch, without the tap tensor: a = (batch, height, width, 64) bf16 NHWC (16-byte aligned),
 * b = the [1][32][64] bf16 tap pack (row (kh*3+kw)*3 + c, column = input channel; 16-byte aligned), sigma optional
 * (device scalar: the taps are divided by it), out = (batch, 3, height, width) fp32.  Bit-identical to
 * ipr_tapgemm_bf16 (linear, IPR_EPI_LINEAR_F32, n_total 32) followed by ipr_col2im3_f32.  One CTA folds whole images
 * in shared memory: height*width must be a multiple of 128 and at most 1024, and width must divide 128
 * (else IPR_E_UNSUPPORTED, and the caller keeps the two-launch path). */
int ipr_tapfold3_f32(const void *a, const void *b, const float *sigma, float *out, int64_t batch, int height,
                     int width, int tanh_out, ipr_stream_t stream);

/* The same layer, same arguments and same results, for larger images: ConvTranspose2d(64,3,3,1,1)+Tanh of
 * networks/conv_generator.py:21-22 and the input gradient of Conv2d(3,64,3,1,1) of networks/sn_discriminator.py:15
 * in the 64 x 64 networks (mg = md = 8), which the entry point above hands back.  A work item is a band of output
 * rows of one image: it stages the taps of its rows and of the rows above and below (recomputed from whole,
 * GEMM-aligned 128-row sub-tiles) and folds them.  Rows per band are chosen per shape (64 x 64: 12).  height*width must be a multiple of 128, width
 * must divide 128 and be at most 128 (else IPR_E_UNSUPPORTED, and the caller keeps the two-launch path); images of
 * 1024 pixels and fewer are accepted too. */
int ipr_tapfold3_band_f32(const void *a, const void *b, const float *sigma, float *out, int64_t batch, int height,
                          int width, int tanh_out, ipr_stream_t stream);

/* BatchNorm2d training-mode statistics (networks/conv_generator.py:9): partial = [rows][2][C] column sums and
 * sums of squares produced by the GEMM epilogue; count = elements per channel.  Writes scale = gamma*rstd,
 * shift = beta - mean*scale, mean, rstd and (if running_mean != NULL) updates the running statistics with
 * `momentum` and the unbiased variance; num_batches_tracked (optional) += 1.  running_* = NULL reproduces
 * DisableBatchNormStats (models/util.py:55-69). */
int ipr_bn_finalize_f32(const float *partial, int rows, int channels, double count, float eps, float momentum,
                        const float *gamma, const float *beta, float *running_mean, float *running_var,
                        int64_t *num_batches_tracked, float *scale, float *shift, float *mean, float *rstd,
                        ipr_stream_t stream);

/* y = relu(x*scale[c] + shift[c]); x, y: [rows][C] bf16 (NHWC). */
int ipr_bn_apply_relu_bf16(const void *x, void *y, const float *scale, const float *shift, int64_t rows,
                           int channels, ipr_stream_t stream);

size_t ipr_bn_bwd_workspace_bytes(int channels);
/* Backward of relu(batchnorm(xraw)) in training mode.  dy, xraw, dx: [rows][C] bf16; scale/shift are the forward's
 * per-channel coefficients (the ReLU mask is recomputed from xraw exactly as the forward evaluated it, so the
 * activation tensor is not re-read).  dgamma / dbeta are written or accumulated.  If sign != NULL the white-box sign-loss
 * gradient  -sign_scale * sign_c / C  (where gamma0 - gamma_c*sign_c > 0) is added to dgamma
 * (tools/sign_model.py:48): the sign loss costs no extra pass. */
int ipr_bn_relu_bwd_bf16(const void *dy, const void *xraw, const float *scale, const float *shift,
                         const float *gamma, const float *mean,
                         const float *rstd, void *dx, float *dgamma, float *dbeta, int accumulate,
                         const float *sign, float gamma0, float sign_scale, void *workspace, size_t workspace_bytes,
                         int64_t rows, int channels, ipr_stream_t stream);

/* Final Linear(K -> 1) of the discriminator (networks/sn_discriminator.py:21): logits[b] = a[b,:].w / sigma + bias.
 * a: [batch][K] bf16, w: fp32 [K] in the activation's (NHWC) feature order. */
int ipr_dfc_fwd_bf16(const void *a, const float *w, const float *sigma, const float *bias, float *logits,
                     int batch, int k, ipr_stream_t stream);
/* da[b,k] = dlogit[b]*w[k]/sigma * (a[b,k] > 0 ? 1 : slope)   (bf16);  dw[j] (+)= sum_b dlogit[b]*a[b,k] (optional),
 * j = dw_index ? dw_index[k] : k (scatter from the NHWC feature order back to the parameter's own order);
 * *dbias += sum_b dlogit[b] (optional, only together with dw; always accumulating, atomically). */
int ipr_dfc_bwd_bf16(const void *a, const float *w, const float *sigma, const float *dlogit, void *da, float *dw,
                     int accumulate_dw, float slope, int batch, int k, const int32_t *dw_index, float *dbias,
                     ipr_stream_t stream);

/* Column sums: out[c] (+)= scale * sum_r in[r*row_stride + c], c < ncols.  `_partials_f32` reduces fp32 partial rows (the GEMM epilogue's
 * per-warp column statistics); `_bf16` reduces an NHWC bf16 tensor over its pixels (bias gradients).
 * Two launches each, fixed summation order (deterministic).  Workspace: ipr_colsum_workspace_bytes(ncols). */
size_t ipr_colsum_workspace_bytes(int ncols);
int ipr_colsum_partials_f32(const float *partial, int rows, int ncols, int row_stride, float *out, int accumulate,
                            float scale, void *workspace, size_t workspace_bytes, ipr_stream_t stream);
/* `_bf16`: out_index (optional) redirects column c to out[out_index[c]]; accumulate == 2 adds atomically (for two
 * producers on different streams: two float contributions onto a zeroed slot are order-independent). */
int ipr_colsum_bf16(const void *x, int64_t rows, int channels, float *out, int accumulate, float scale,
                    const int32_t *out_index, void *workspace, size_t workspace_bytes, ipr_stream_t stream);

/* ------------------------------------------------------------------ spectral norm, optimizer, weight packing */

#define IPR_SN_MAX_LAYERS 16
typedef struct {
    const float *w;        /* fp32 master weight viewed as (rows, cols) row-major (weight_orig)            */
    float *u, *v;          /* power-iteration vectors (weight_u: rows, weight_v: cols), updated in place     */
    float *sigma;          /* device scalar written by the power iteration, read by the weight gradient     */
    float *grad;           /* ipr_sn_weight_grad_f32: gradient w.r.t. W/sigma in, w.r.t. W out (in place)   */
    float *grad_out;       /* optional: if not NULL the result is ADDED here instead (e.g. the .grad arena)   */
    int32_t rows, cols;
    int64_t scratch_off;   /* offset (floats) of this layer's private slice of `scratch`,
                              at least ipr_sn_scratch_floats(rows, cols) long                               */
    float *u_snap, *v_snap; /* optional: ipr_sn_power_iter_f32 also writes the vectors it leaves in u / v here
                              (the copy one forward keeps for its backward while the buffers move on)        */
} ipr_sn_layer_t;

size_t ipr_sn_scratch_floats(int rows, int cols);
/* One power iteration for every layer (update != 0; training forward) or just sigma = u.(W v) (update == 0; eval),
 * exactly as torch.nn.utils.spectral_norm does per layer and per forward (networks/sn_discriminator.py:1). */
int ipr_sn_power_iter_f32(const ipr_sn_layer_t *layers_host, int n_layers, int update, float eps, float *scratch,
                          ipr_stream_t stream);
/* grad <- (grad - <grad, W>/sigma * u v^T) / sigma for every layer: backward of W -> W / sigma(W). */
int ipr_sn_weight_grad_f32(const ipr_sn_layer_t *layers_host, int n_layers, float *scratch, ipr_stream_t stream);

/* Adam (torch.optim.Adam semantics, models/dcgan.py:21-24) over flat fp32 arenas in one launch; *step (device
 * float) is read then incremented on the device, so the call is CUDA-graph replayable. */
/* grad_scale multiplies every gradient element first (1/world after a summing all-reduce); zero_grad != 0 clears
 * the gradient arena as it is consumed (the next step's optimizer.zero_grad() then has nothing left to do);
 * *ticket is a zero-initialised device word the launch uses to publish step + 1 once every CTA has read step. */
int ipr_adam_flat_f32(float *param, float *grad, float *exp_avg, float *exp_avg_sq, int64_t n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, float grad_scale, int zero_grad,
                      float *step, uint32_t *ticket, ipr_stream_t stream);

/* dst[i] = bf16(index[i] >= 0 ? src[index[i]] : 0), n % 8 == 0: rebuilds every GEMM operand layout of a network
 * from its fp32 parameter arena in one launch. */
/* The same launch also fills an fp32 side table dst_f32[i] = src[index_f32[i]] (n_f32 may be 0): permuted copies of
 * the few parameters kernels read in fp32 (Linear bias in NHWC feature order, the final GEMV row). */
int ipr_gather_pack_bf16(const float *src, const int32_t *index, void *dst, int64_t n, const int32_t *index_f32,
                         float *dst_f32, int64_t n_f32, ipr_stream_t stream);

/* ---- scalar ends of the step (csrc/step_misc.cu) ------------------------------------------------------------
 * Hinge discriminator loss (models/dcgan.py:31-35): losses[0..2] = LossD, LossR, LossF with
 * LossR = mean relu(1 - real), LossF = mean relu(1 + fake); d_real / d_fake (optional) = dLossD/dlogits.
 * Stored losses are multiplied by loss_scale (gradients are not), see ipr_ssim_fwd_bwd_f32. */
int ipr_hinge_d_loss_f32(const float *real_logits, const float *fake_logits, int batch, float loss_scale,
                         float *losses, float *d_real, float *d_fake, ipr_stream_t stream);
/* Generator adversarial loss (models/dcgan.py:37-40): *loss = -mean(logits); dlogits (optional) = -1/batch. */
int ipr_gen_adv_loss_f32(const float *logits, int batch, float loss_scale, float *loss, float *dlogits,
                         ipr_stream_t stream);
/* Pointwise losses of the SRGAN / CycleGAN steps, value and gradient in one pass over x:
 *   kind 0  mean (x-y)^2   (F.mse_loss, nn.MSELoss: models/srgan.py:49,59, models/cyclegan.py:122-143)
 *   kind 1  mean |x-y|     (nn.L1Loss: models/cyclegan.py:125-133)
 *   kind 2  mean BCE-with-logits (models/srgan.py:36-56)
 * y == NULL: the target is the constant y0.  *loss = weight * mean(...), dx (optional) = weight * d mean / dx.
 * Fixed-order two-stage reduction (deterministic). */
size_t ipr_pointwise_loss_workspace_bytes(void);
int ipr_pointwise_loss_f32(const float *x, const float *y, float y0, int64_t n, int kind, float weight, float *loss,
                           float *dx, void *workspace, size_t workspace_bytes, ipr_stream_t stream);
/* n standard-normal draws (Philox4x32-10 keyed by seed, Box-Muller); *counter (device) is the stream position and
 * advances by ceil(n/4) per launch, *ticket a zero-initialised device word: graph-replayable latent generation
 * replacing the host-side torch.randn + H2D copy of experiments/image_generation.py:94. */
int ipr_randn_f32(float *out, int64_t n, uint64_t seed, uint64_t *counter, uint32_t *ticket, ipr_stream_t stream);

/* ------------------------------------------------------------------ generic layers (csrc/layers.cu)
 * The SRGAN / CycleGAN network families (networks/sr_resnet.py:3-44, discriminator_96.py:3-35,
 * resnet_generator.py:3-59, conv_discriminator.py:3-21): a convolution of any of their shapes is
 *   ipr_im2col_nhwc_bf16 (patch matrix)  ->  ipr_tapgemm_bf16 (single-tap "linear" GEMM on tcgen05),
 * its data gradient  ipr_tapgemm_bf16 (dY x W^T)  ->  ipr_col2im_nhwc_bf16 (adjoint gather),
 * its weight gradient  ipr_wgrad_bf16 (dY^T x patch matrix).
 *
 * Patch matrix of an NHWC bf16 tensor x (n,h,w,c; c % 8 == 0):
 *   col[(img, oy, ox)][(ky*k + kx)*c + ch] = x[img, src(oy*stride + ky - pad), src(ox*stride + kx - pad), ch]
 * rows are kp elements long (kp % 8 == 0, kp >= k*k*c, the tail is zero).  src(): zero outside the image, or
 * (reflect != 0) mirrored without repeating the edge (nn.ReflectionPad2d); up > 1 runs a transposed convolution
 * as a direct one over the zero-inserted grid (coordinates not divisible by up, or past (size-1)*up, read zero). */
int ipr_im2col_nhwc_bf16(const void *x, void *col, int n, int h, int w, int c, int oh, int ow, int k, int stride,
                         int pad, int up, int reflect, int kp, ipr_stream_t stream);
/* Adjoint of the above: dx[img, iy, ix, ch] = addend (optional, same shape) + sum of every dcol entry that read it. */
int ipr_col2im_nhwc_bf16(const void *dcol, void *dx, const void *addend, int n, int h, int w, int c, int oh, int ow,
                         int k, int stride, int pad, int up, int reflect, int kp, ipr_stream_t stream);
/* Module boundary: NCHW fp32 -> NHWC bf16 with channels zero-padded to cp (cp % 8 == 0); tanh_out (optional, same
 * shape as x) multiplies by 1 - tanh_out^2 (backward of a final Tanh fused into the gradient's layout change). */
int ipr_nchw_to_nhwc_bf16(const float *x, const float *tanh_out, void *y, int64_t n, int c, int h, int w, int cp,
                          ipr_stream_t stream);
/* fp32 GEMM result t[pixel][ld] (+ bias[ch], optional) -> NCHW fp32 (first c columns), optional Tanh. */
int ipr_finish_nchw_f32(const float *t, const float *bias, float *out, int64_t n, int c, int h, int w, int ld,
                        int tanh_out, ipr_stream_t stream);
/* nn.PixelShuffle(2) on NHWC bf16: y[n,2h+i,2w+j,c] = x[n,h,w,c*4+i*2+j] (inverse != 0: x is the large grid). */
int ipr_pixel_shuffle2_nhwc_bf16(const void *x, void *y, int64_t n, int h, int w, int c_out, int inverse,
                                 ipr_stream_t stream);
int ipr_add_bf16(const void *a, const void *b, void *out, int64_t n, ipr_stream_t stream);

/* Normalisation (+ activation, + residual) over an NHWC bf16 tensor viewed as [groups][rows][channels]:
 * groups = 1 is BatchNorm2d in training mode (statistics over all rows; running statistics and
 * num_batches_tracked updated when given), groups = batch is InstanceNorm2d (per image).
 * has_norm: 0 = activation only, 1 = normalise with the statistics of x, 2 = normalise with the given
 * scale / shift (eval-mode BatchNorm).  scale/shift/mean/rstd: [groups][channels] outputs kept for the backward.
 * act: 0 none, 1 ReLU, 2 LeakyReLU(slope), 3 PReLU (single parameter, read from slope_ptr), 4 Tanh.
 * y = act(x * scale + shift) + residual (optional).  gamma / beta NULL = non-affine. */
size_t ipr_norm_workspace_bytes(int groups, int channels);
int ipr_norm_fwd_bf16(const void *x, void *y, const void *residual, int groups, int64_t rows, int channels,
                      int has_norm, float eps, float momentum, const float *gamma, const float *beta,
                      float *running_mean, float *running_var, int64_t *num_batches_tracked, float *scale,
                      float *shift, float *mean, float *rstd, int act, float slope, const float *slope_ptr,
                      void *workspace, size_t workspace_bytes, ipr_stream_t stream);
/* Backward of the above (x = the forward's raw input): dx; dgamma / dbeta (+)= (optional); *dslope (+)= PReLU slope
 * gradient (optional).  sign != NULL adds the white-box sign-loss gradient
 * -sign_scale * sign_c / channels * [gamma0 - gamma_c*sign_c > 0] to dgamma (tools/sign_model.py:42-49), for
 * BatchNorm and InstanceNorm alike. */
int ipr_norm_bwd_bf16(const void *dy, const void *x, void *dx, int groups, int64_t rows, int channels, int has_norm,
                      const float *gamma, const float *scale, const float *shift, const float *mean,
                      const float *rstd, float *dgamma, float *dbeta, int accumulate, const float *sign, float gamma0,
                      float sign_scale, int act, float slope, const float *slope_ptr, float *dslope, void *workspace,
                      size_t workspace_bytes, ipr_stream_t stream);

/* ------------------------------------------------------------------ robustness attacks (csrc/prune.cu)
 * Global magnitude pruning, in place, over the N = n_total entries of a list of segments of an fp32 parameter
 * arena: the removal attack of the reference's prune.py (SURVEY.md 2.1 row 34), i.e.
 * torch.nn.utils.prune.global_unstructured(..., pruning_method=L1Unstructured, amount) with k = round(amount * N).
 *   segments: device table of n_segments (offset, count) int64 pairs, offsets ascending, segments disjoint,
 *             counts > 0 summing to n_total (8-byte aligned; n_segments <= IPR_PRUNE_MAX_SEGMENTS);
 *   exactly k entries are zeroed, those with the smallest |w| over all segments together; a zeroed entry becomes
 *   w * 0 (a negative weight becomes -0.0: bit-identical to weight_orig * weight_mask); +-0 share the key 0 and
 *   every NaN ranks above every finite value and +inf (torch.topk's order);
 *   ties at the k-th magnitude, whose order torch leaves unspecified: the lowest arena index is pruned first;
 *   k = 0 launches nothing, k = N zeroes every segment entry; entries outside the segments are never written.
 * The threshold is selected on the device (radix select), nothing is read back: the launches are graph-capturable.
 * workspace: ipr_prune_workspace_bytes(n_total) bytes, 256-byte aligned. */
#define IPR_PRUNE_MAX_SEGMENTS 256
size_t ipr_prune_workspace_bytes(int64_t n_total);
int ipr_prune_magnitude_f32(float *arena, const int64_t *segments, int n_segments, int64_t n_total, int64_t k,
                            void *workspace, size_t workspace_bytes, ipr_stream_t stream);
/* arena[index[i]] = -arena[index[i]] for i < n, indices distinct (device int64 list): the sign flip of
 * normalisation gammas of the ambiguity attack (sign_flip.py:59-77).  One launch; n = 0 launches nothing. */
int ipr_negate_indexed_f32(float *arena, const int64_t *index, int64_t n, ipr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* IPR_B200_H */
