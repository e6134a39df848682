/* b200seg.h — C ABI of libb200seg.so: the sm_100a kernels behind the drop-in U-Net-family modules.
 *
 * The reference (bababyVN/medical-image-segmentation-and-classification) is pure Python and has NO FFI /
 * plugin layer: its boundary for this path is the nn.Module surface, and every entry point below replaces the
 * ATen/cuDNN op that a reference module line dispatches to.  Each declaration cites that call site
 * (file:line relative to the reference root).  INTEGRATION.md shows the ctypes / torch.library binding.
 *
 * Conventions
 *   - plain pointers + sizes; all pointers are DEVICE pointers owned by the caller (PyTorch allocates them);
 *   - activations are NHWC bf16; `ld*` is the channel stride in ELEMENTS of the underlying buffer, so a channel
 *     slice of a wider buffer can be passed without a copy;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), never allocates, never syncs;
 *   - return 0 on success or a negative B2_ERR_* code; b2_last_error() gives the thread-local message;
 *   - no CPU fallback, no cuDNN/cuBLAS: on a non-sm_100 device every compute entry returns B2_ERR_ARCH.
 */
#ifndef B200SEG_H_
#define B200SEG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2_ABI_VERSION 1

enum {
  B2_OK = 0,
  B2_ERR_SHAPE = -1,     /* unsupported / inconsistent dimensions */
  B2_ERR_ALIGN = -2,     /* pointer or stride alignment (16 B) violated */
  B2_ERR_ARCH = -3,      /* device is not sm_100 (B200) */
  B2_ERR_CUDA = -4,      /* CUDA runtime / driver error */
  B2_ERR_NCCL = -5,      /* reserved for the collective path */
  B2_ERR_WORKSPACE = -6  /* caller-provided workspace too small */
};

typedef void* b2_stream_t; /* cudaStream_t */

const char* b2_last_error(void);
int b2_abi_version(void);
int b2_arch_check(void);   /* 0 iff the current device is sm_100; B2_ERR_ARCH otherwise */
int b2_num_sms(void);

/* Deterministic-reduction mode (SURVEY.md §5 / §7.2-4: cuDNN's BatchNorm in the reference, AttentionUNet.py:7, is
 * run-to-run reproducible; fp64/fp32 atomics are not).  With a workspace registered for the current device every
 * kernel that would end in cross-block atomics — the BatchNorm statistics of the conv epilogue, the BatchNorm /
 * gate backward sums, bias and head gradients, the loss sums, the gradient norm — writes one row of per-block
 * partials into it and a second tiny kernel adds the rows in block order, so two runs on the same inputs are
 * bit-identical.  The workspace (>= 1 MiB, 64 MiB covers every shape of the four models) is used by the launches
 * of ONE compute stream at a time; NULL switches the mode off.  b2_get_deterministic() -> 0 | 1. */
int b2_set_deterministic(void* workspace, int64_t bytes);
int b2_get_deterministic(void);
/* The finish of that mode on its own: for each segment k < nseg (1..4), dsts[k][i] += the sum over the rows
 * r = 0, 1, ..., rows-1, in that order and in fp64, of partial[r * row_stride + offsets[k] + i], for i < counts[k];
 * dsts[k] is double when dst_f64[k] != 0 and float otherwise.  One launch for all segments. */
int b2_det_finish(const double* partial, int64_t rows, int32_t row_stride, int32_t nseg, const int32_t* offsets,
                  const int32_t* counts, void* const* dsts, const int32_t* dst_f64, b2_stream_t stream);

/* The B200SEG_* environment switches (DESIGN.md section 10) are read once and cached behind a mutex; call this after
 * changing the environment of a running process (tests do) to have them re-read. */
int b2_reload_env(void);

/* ------------------------------------------------------------------------------------------------------------
 * Convolution, ksize in {1,3} with 'same' padding (stride 1 or 2) or ksize 2 / stride 2 / no padding (the input
 * gradient of ConvTranspose2d(k=2,s=2)): implicit GEMM on tcgen05 (TMA -> 128B-swizzled smem ->
 * tcgen05.mma, fp32 accumulators in TMEM).  Replaces nn.Conv2d forward at
 *   models/segmentation_models/AttentionUNet.py:6,9,20,33,37,41   R2U_Net.py:10,27,43   R2AttU_Net.py:35,52,65-74
 *   ResnetUnet.py:7,10,54
 * and, run on dgrad-packed weights (b2_pack_weights), the input-gradient half of aten::convolution_backward
 * (autograd of utils/helpers.py:329).
 * The K dimension may come from two tensors (x0 | x1): this is the elided torch.cat of AttentionUNet.py:101,106,
 * 111,116 / R2U_Net.py:94.. .  Epilogue: +bias, +addend (bf16 residual), optional ReLU, bf16 store, and
 * per-channel sum / sum-of-squares of the ROUNDED output accumulated into `stats` (BatchNorm batch statistics,
 * AttentionUNet.py:7,10,21).
 * Requirements: c0,c1 multiples of 8 (c0 multiple of 64 when c1 > 0); cout multiple of 32; W a power of two >= 8
 * or a multiple of 128, H*W..: see DESIGN.md "tile geometry".
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_conv_args {
  int32_t n, h, w;        /* output == input spatial extent */
  int32_t ksize;          /* 1 or 3 */
  const void* x0;         /* NHWC bf16 */
  int32_t c0, ldx0;
  const void* x1;         /* optional second K source (NULL if unused) */
  int32_t c1, ldx1;
  const void* wpk;        /* packed bf16 [ksize*ksize][rows][ktot], rows >= cout */
  int32_t ktot;           /* row length of wpk in elements (>= c0 + c1) */
  int64_t w_tap_stride;   /* elements between taps in wpk */
  int32_t cout;
  void* y;                /* NHWC bf16 */
  int32_t ldy;
  const float* bias;      /* [cout] or NULL */
  const void* addend;     /* optional NHWC bf16 [.., cout] added before rounding (NULL if unused) */
  int32_t ldadd;
  double* stats;          /* optional [2][cout] (sum, sumsq), ACCUMULATED into (caller zeroes) */
  int32_t relu;
  /* extensions (0 = default): input sampling stride (1|2; the input extent is then h*stride x w*stride) and a
   * strided output placement y[n, h*out_mul + out_off_h, w*out_mul + out_off_w, :] inside an (h*out_mul) x
   * (w*out_mul) image — the pixel-shuffle scatter of ConvTranspose2d(k=2,s=2) (ResnetUnet.py:21,53) */
  int32_t stride;
  int32_t out_mul, out_off_h, out_off_w;
  /* the A operand may likewise be the sub-lattice x[n, h*in_mul + in_off_h, w*in_mul + in_off_w, :] of an
   * (h*in_mul) x (w*in_mul) image, and the tap offsets (r - pad_h, s - pad_w) may be overridden (custom_pad != 0):
   * the four 2x2 phase convolutions that nearest-x2 upsampling + conv3x3 decomposes into (UpConv,
   * AttentionUNet.py:15-27) are expressed with ksize 2, custom pads and these placements */
  int32_t in_mul, in_off_h, in_off_w;
  int32_t custom_pad, pad_h, pad_w;
  int32_t add_after_act;  /* 1: y = act(conv + bias) + addend (Recurrent_block's x + x1 in the folded inference path) */
  /* merged launches of the folded UpConv (ksize 2; wpk = the 16 packed taps [4 phases][4 taps][rows][ktot]):
   *   1 = fprop:  x0 is the coarse input [n, h, w, c0], y the FINE output [n, 2h, 2w, cout] — all four phase
   *               convolutions in one launch (phase = extra tile dimension, pixel-shuffle stores);
   *   2 = dgrad:  x0 is the FINE gradient dz [n, 2h, 2w, c0], y the coarse dx [n, h, w, cout] — the four phases are
   *               one K loop of 16 taps over the sub-lattices of dz (no addend chain). */
  int32_t fold_mode;
} b2_conv_args;

int b2_conv_fprop(const b2_conv_args* a, b2_stream_t stream);
/* same kernel; `wpk` must be the dgrad packing, x0 is dY, y is dX */
int b2_conv_dgrad(const b2_conv_args* a, b2_stream_t stream);

/* Weight gradient: dW[co][tap][ci] = sum_p dY[p][co] * X[p (+) tap][ci]  (the weight half of
 * aten::convolution_backward).  tcgen05 with MN-major operands, split-K over pixels, deterministic two-stage
 * reduction through `workspace`.  dw is fp32 laid out [cout][ksize*ksize][c0+c1] (== channels_last weight). */
typedef struct b2_wgrad_args {
  int32_t n, h, w;
  int32_t ksize;
  const void* dy;         /* NHWC bf16 */
  int32_t cout, lddy;
  const void* x0;
  int32_t c0, ldx0;
  const void* x1;
  int32_t c1, ldx1;
  float* dw;
  int32_t accumulate;     /* 1: dw += result (shared weights of R2U_Net.py:15-20), 0: overwrite */
  void* workspace;
  int64_t workspace_bytes;
  /* extension (0 = 1): sampling stride of the X operand; 2 with ksize 2 computes the weight gradient of
   * ConvTranspose2d(k=2,s=2) (dy := the transposed conv's INPUT on the coarse grid, x := its output gradient on the
   * 2x grid; result [cin_T][2*2][cout_T]) */
  int32_t x_stride;
  /* dY as the sub-lattice dy[n, h*dy_mul + dy_off_h, w*dy_mul + dy_off_w, :]; custom X tap offsets (see b2_conv_args) */
  int32_t dy_mul, dy_off_h, dy_off_w;
  int32_t custom_pad, pad_h, pad_w;
  /* extension (0 = off): merged weight gradient of a folded UpConv (Upsample x2 -> conv3x3, AttentionUNet.py:15-27).
   * ksize 2, dy_mul 2, no offsets: dy is the gradient on the FINE grid [n, 2h, 2w, cout], x the coarse input, and
   * dw receives all four phase gradients [phase = 2a + b][cout][2x2][cin] (phase (a,b): dy[2h+a, 2w+b] against
   * x[h + a + ty - 1, w + b + tx - 1]) from ONE launch instead of four dy_off launches.  cout must be 64 or a
   * multiple of 128, cin a multiple of 64, the coarse image at least 16 pixels wide (B2_ERR_SHAPE otherwise). */
  int32_t fold;
} b2_wgrad_args;

int64_t b2_conv_wgrad_workspace(const b2_wgrad_args* a);
int b2_conv_wgrad(const b2_wgrad_args* a, b2_stream_t stream);

/* fp32 [cout][cin][k][k] parameter with arbitrary element strides -> bf16 fprop packing [k*k][cout][cin] and
 * (optional) dgrad packing [k*k][cin][cout] with the taps flipped. */
int b2_pack_weights(const float* w, int32_t cout, int32_t cin, int32_t ksize, int64_t s_co, int64_t s_ci,
                    int64_t s_kh, int64_t s_kw, void* w_fprop, void* w_dgrad, b2_stream_t stream);

/* Inference (eval-mode) BatchNorm folding, Appendix D.3 of SURVEY.md: W' = W * scale[co] packed for fprop (plain, or
 * the 16-tap UpConv folding when upfold != 0) and b' = bias * scale + shift, so that conv + BN + ReLU is ONE tcgen05
 * launch with a bias/ReLU epilogue (pipeline.py:340-357 / tester.py:264-289 inference path). */
int b2_pack_weights_folded(const float* w, int32_t cout, int32_t cin, int32_t ksize, int64_t s_co, int64_t s_ci,
                           int64_t s_kh, int64_t s_kw, const float* scale, const float* shift, const float* bias,
                           int32_t upfold, void* w_fprop, float* bias_out, b2_stream_t stream);

/* UpConv folding (AttentionUNet.py:15-27: nearest x2 upsample followed by conv3x3): phase (a,b) of the 2x output grid
 * is a 2x2 convolution of the LOW-resolution input with weights W_ab[u][v] = sum_{r in R_a(u)} sum_{s in R_b(v)} W[r][s],
 * R_0 = ({0},{1,2}), R_1 = ({0,1},{2})  — 2.25x fewer FLOPs, exact algebra.
 * w_fprop: bf16 [4 phases][4 taps][cout][cin];  w_dgrad: bf16 [4 phases][4 taps flipped][cin][cout] (may be NULL) */
int b2_pack_weights_upfold(const float* w, int32_t cout, int32_t cin, int64_t s_co, int64_t s_ci, int64_t s_kh,
                           int64_t s_kw, void* w_fprop, void* w_dgrad, b2_stream_t stream);
/* adjoint of the folding: dw[cout][9][cin] = scatter-sum of dweff[4 phases][cout][4 taps][cin] (fp32) */
int b2_fold_upconv_wgrad(const float* dweff, int32_t cout, int32_t cin, float* dw, b2_stream_t stream);

/* Small-Cin direct convolution (image stem: AttentionUNet.py:6 with cin=3, R2U_Net.py:43 RRCNN1.conv_1x1).
 * x is NHWC bf16 padded to 4 channels; w is fp32 [cout][ksize*ksize][4]. */
int b2_conv_smallc_fprop(const void* x4, int32_t n, int32_t h, int32_t w, int32_t ksize, const float* wk,
                         const float* bias, int32_t cout, void* y, int32_t ldy, int32_t relu, b2_stream_t stream);
int b2_conv_smallc_wgrad(const void* dy, int32_t lddy, const void* x4, int32_t n, int32_t h, int32_t w,
                         int32_t ksize, int32_t cout, float* dw /* [cout][k*k][4], accumulated into */,
                         b2_stream_t stream);

/* Cout<=8 1x1 heads (AttentionUNet.py:84, R2U_Net.py:76, ResnetUnet.py:58): memory-bound dot products.
 * y is fp32 NCHW [n][cout][hw]; x NHWC bf16. */
int b2_head_fwd(const void* x, int32_t ldx, int64_t npix, int32_t hw, int32_t cin, const float* w /*[cout][cin]*/,
                const float* bias, int32_t cout, float* y, b2_stream_t stream);
int b2_head_bwd(const float* dy, const void* x, int32_t ldx, int64_t npix, int32_t hw, int32_t cin,
                const float* w, int32_t cout, void* dx, int32_t lddx, float* dw /*accumulated*/,
                float* db /*accumulated*/, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * BatchNorm2d (AttentionUNet.py:7,10,21,34,38,42; R2U_Net.py:11,28; ResnetUnet.py:8,11,55), eps/momentum as args.
 * ---------------------------------------------------------------------------------------------------------- */
int b2_channel_stats(const void* z, int32_t ldz, int64_t npix, int32_t c, double* stats, b2_stream_t stream);
/* mean/invstd/scale/shift may all be NULL (running-statistics update only); running_* / nbt may be NULL */
int b2_bn_finalize(const double* stats, int32_t c, int64_t count, const float* gamma, const float* beta,
                   float eps, float momentum, float* running_mean, float* running_var,
                   int64_t* num_batches_tracked, float* mean, float* invstd, float* scale, float* shift,
                   b2_stream_t stream);
/* The running-statistics half of b2_bn_finalize (momentum update with the unbiased variance, num_batches_tracked += 1;
 * nn.BatchNorm2d semantics, AttentionUNet.py:7) for MANY layers in one launch: a training step of AttU_Net has 34
 * BatchNorm calls whose updates are off the data path, so the step queues them and flushes once.  `refs` is a HOST
 * array of n entries (they travel to the device as kernel parameters, 64 per launch: nothing to keep alive, safe
 * under CUDA-graph capture); the entries of one call must refer to DISTINCT layers; max_c = the largest channel count. */
typedef struct b2_bn_run_ref {
  const double* stats;             /* [2][c]: sum, sum of squares */
  float* running_mean;
  float* running_var;
  int64_t* num_batches_tracked;
  int64_t count;                   /* elements per channel */
  int32_t c;
  float momentum;
} b2_bn_run_ref;
int b2_bn_update_running_multi(const b2_bn_run_ref* refs, int32_t n, int32_t max_c, b2_stream_t stream);
int b2_bn_eval_coeffs(const float* gamma, const float* beta, const float* running_mean,
                      const float* running_var, float eps, int32_t c, float* mean, float* invstd, float* scale,
                      float* shift, b2_stream_t stream);
/* y = act(z*scale+shift) ; with ysum: also ysum = y + addend (Recurrent_block's x + x1, R2U_Net.py:19);
 * with addend but ysum == NULL: y = act(z*scale+shift + addend) (torchvision Bottleneck residual) */
int b2_bn_apply(const void* z, int32_t ldz, int64_t npix, int32_t c, const float* scale, const float* shift,
                int32_t relu, void* y, int32_t ldy, const void* addend, int32_t ldadd, void* ysum,
                int32_t ldysum, b2_stream_t stream);
/* sums[0][c] = sum dy*mask ; sums[1][c] = sum dy*mask*xhat   (caller zeroes) */
int b2_bn_bwd_reduce(const void* dy, int32_t lddy, const void* z, int32_t ldz, int64_t npix, int32_t c,
                     const float* scale, const float* shift, const float* mean, const float* invstd,
                     int32_t relu, double* sums, b2_stream_t stream);
/* dz = gamma*invstd*(dy*mask - [training](sums0/m + xhat*sums1/m)); also writes dgamma/dbeta (fp32) and, if
 * dbias != NULL, accumulates dbias[c] += sum_p dz[p][c] (bias gradient of the producing conv; caller zeroes) */
int b2_bn_bwd_apply(const void* dy, int32_t lddy, const void* z, int32_t ldz, int64_t npix, int32_t c,
                    const float* scale, const float* shift, const float* mean, const float* invstd,
                    const float* gamma, int32_t relu, int32_t training, const double* sums, void* dz,
                    int32_t lddz, float* dgamma, float* dbeta, float* dbias, b2_stream_t stream);
/* db[c] = sum_p dy[p][c] (bias gradient of a conv; overwrite) */
int b2_channel_sum(const void* dy, int32_t lddy, int64_t npix, int32_t c, float* db, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Pooling / upsampling / elementwise (AttentionUNet.py:61,18; R2U_Net.py:54,25,19,48)
 * ---------------------------------------------------------------------------------------------------------- */
int b2_maxpool2x2_fwd(const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w, int32_t c, void* y,
                      int32_t ldy, b2_stream_t stream);
int b2_maxpool2x2_bwd(const void* dy, int32_t lddy, const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w,
                      int32_t c, void* dx, int32_t lddx, b2_stream_t stream);
/* dx = maxpool gradient + addend: the skip tensor of a U-Net level has two consumers (the pool, AttentionUNet.py:88-94,
 * and the decoder's gate / concat, :100-101); taking the decoder-side gradient as the addend replaces autograd's
 * separate full-size accumulation (one rounding, as ATen's add of the two bf16 gradients). */
int b2_maxpool2x2_bwd_add(const void* dy, int32_t lddy, const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w,
                          int32_t c, const void* addend, int32_t ldadd, void* dx, int32_t lddx, b2_stream_t stream);
int b2_upsample2x_fwd(const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w, int32_t c, void* y,
                      int32_t ldy, b2_stream_t stream);
int b2_upsample2x_bwd(const void* dy, int32_t lddy, int32_t n, int32_t h, int32_t w, int32_t c, void* dx,
                      int32_t lddx, b2_stream_t stream);
int b2_add(const void* a, int32_t lda, const void* b, int32_t ldb, int64_t npix, int32_t c, void* out,
           int32_t ldo, b2_stream_t stream);
int b2_nchw_f32_to_nhwc_bf16(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, void* y, int32_t ldy,
                             b2_stream_t stream);
/* module-boundary adapters for any channel count (input arrives NCHW fp32: utils/helpers.py:318) */
/* Image stem as a GEMM (AttentionUNet.py:6 basic_block(3,64) first conv, K = 27): xc[N,H,W,32] bf16 = im2col of the
 * 3x3 neighbourhood of the fp32 NCHW image x[N,c<=3,H,W] (column = tap*c_in + channel, zero padded to 32), consumed by
 * b2_conv_fprop / b2_conv_wgrad as a 1x1 convolution with 32 input channels. */
int b2_stem_im2col3x3(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, void* xc, b2_stream_t stream);
int b2_layout_nchw_to_nhwc(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, void* y, int32_t ldy,
                           b2_stream_t stream);
int b2_layout_nhwc_to_nchw(const void* x, int32_t ldx, int32_t n, int32_t c, int32_t h, int32_t w, float* y,
                           b2_stream_t stream);

/* ResNet-50 encoder of ResNetUnet (ResnetUnet.py:32-43), forward only (frozen by default):
 * 7x7/s2/p3 stem conv 3->64 without bias (x4 = NHWC bf16 padded to 4 channels, wk fp32 [64][49][4]) and
 * MaxPool2d(3, 2, 1); h, w are INPUT extents */
int b2_stem7x7_fprop(const void* x4, int32_t n, int32_t h, int32_t w, const float* wk, int32_t cout, void* y,
                     int32_t ldy, b2_stream_t stream);
int b2_maxpool3x3s2_fwd(const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w, int32_t c, void* y,
                        int32_t ldy, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Attention gate (AttentionUNet.py:48-54, R2AttU_Net.py:80-86) — the 1x1 GEMMs go through b2_conv_fprop.
 * ---------------------------------------------------------------------------------------------------------- */
/* a = relu(bf16(bn_g(g1p)) + bf16(bn_x(x1p))); q = a . wpsi + bpsi (bf16) ; qstats += (sum q, sum q^2) */
int b2_gate_psi_fwd(const void* g1p, const void* x1p, int32_t ld, int64_t npix, int32_t fint,
                    const float* scale_g, const float* shift_g, const float* scale_x, const float* shift_x,
                    const float* wpsi, const float* bpsi, void* q, double* qstats, b2_stream_t stream);
/* psi = sigmoid(bn1(q)) ; out = x * psi */
int b2_gate_apply_fwd(const void* x, int32_t ldx, const void* q, int64_t npix, int32_t c, const float* scale1,
                      const float* shift1, void* psi, void* out, int32_t ldo, b2_stream_t stream);
/* dx = dout*psi ; dsig[p] = (sum_c dout*x) * psi*(1-psi) ; sums1 += (sum dsig, sum dsig*qhat) */
int b2_gate_apply_bwd(const void* dout, int32_t lddout, const void* x, int32_t ldx, const void* psi,
                      const void* q, int64_t npix, int32_t c, const float* mean1, const float* invstd1,
                      void* dx, int32_t lddx, float* dsig, double* sums1, b2_stream_t stream);
/* per-channel coefficient pointers of the three BatchNorms inside a gate + the psi weight (all device fp32) */
typedef struct b2_gate_coef {
  const float *scale_g, *shift_g, *mean_g, *invstd_g, *gamma_g;   /* W_g.1 : [fint] */
  const float *scale_x, *shift_x, *mean_x, *invstd_x, *gamma_x;   /* W_x.1 : [fint] */
  const float *gamma1, *mean1, *invstd1;                          /* psi.1 : [1]    */
  const float* wpsi;                                              /* psi.0.weight : [fint] */
} b2_gate_coef;
/* dq from dsig (BN1 backward), da = dq*wpsi*(a>0); reductions for both inner BNs and the psi conv:
 * sums[0..3][fint] = dbeta_g, dgamma_g, dbeta_x, dgamma_x (fp64, caller zeroes);
 * dwpsi[fint], dbpsi[1] fp32, accumulated into (caller zeroes) */
int b2_gate_psi_bwd_reduce(const float* dsig, const void* q, const void* g1p, const void* x1p, int32_t ld,
                           int64_t npix, int32_t fint, const b2_gate_coef* coef, const double* sums1,
                           int32_t training, double* sums, float* dwpsi, float* dbpsi, b2_stream_t stream);
/* dg1p, dx1p (bf16 [npix][fint]); dgamma_beta fp32 [4][fint] = dgamma_g, dbeta_g, dgamma_x, dbeta_x;
 * dbn1 fp32 [2] = dgamma1, dbeta1; dbias (optional, fp32 [2][fint], accumulated, caller zeroes) = column sums of
 * dg1p / dx1p = bias gradients of the W_g / W_x convolutions */
int b2_gate_psi_bwd_apply(const float* dsig, const void* q, const void* g1p, const void* x1p, int32_t ld,
                          int64_t npix, int32_t fint, const b2_gate_coef* coef, const double* sums1,
                          int32_t training, const double* sums, void* dg1p, void* dx1p, float* dgamma_beta,
                          float* dbn1, float* dbias, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Loss: BCEWithLogits (utils/helpers.py:245,327) and 0.5*BCE + 0.5*Dice (utils/clip_seg_finetuner.py:40-74)
 * sums[6] = sum bce_i, sum sigmoid(z)*t, sum sigmoid(z), sum t, #(pred&t), #(pred|t) with pred = z>0 (caller zeroes;
 * the last two are the IoU counts of utils/helpers.py:223-227 at threshold 0.5)
 * ---------------------------------------------------------------------------------------------------------- */
int b2_loss_fwd(const float* z, const float* t, int64_t count, double* sums, b2_stream_t stream);
/* loss = w_bce * sums[0]/count + w_dice * (1 - (2*sums[1]+smooth)/(sums[2]+sums[3]+smooth)) */
int b2_loss_finalize(const double* sums, int64_t count, float w_bce, float w_dice, float smooth, float* loss,
                     b2_stream_t stream);
/* dz = grad_out * d loss / d z */
int b2_loss_bwd(const float* z, const float* t, int64_t count, const double* sums, float w_bce, float w_dice,
                float smooth, const float* grad_out, float* dz, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Validation / test metrics and the served mask (SURVEY.md section 8f, N2 / N3)
 * counts[n][3] = {TP, #pred, #target} per sample with pred = z > thr_logit (== sigmoid(z) > threshold,
 * thr_logit = log(thr / (1 - thr))) and target = t > thr_target: the integers behind calculate_iou / calculate_dice /
 * calculate_pixel_accuracy / calculate_segmentation_metrics (utils/tester.py:92-193) and iou (utils/helpers.py:223-227).
 * The library zeroes counts. z, t: [n][per_sample] fp32 contiguous.
 * ---------------------------------------------------------------------------------------------------------- */
int b2_seg_counts(const float* z, const float* t, int32_t n, int64_t per_sample, float thr_logit, float thr_target,
                  uint64_t* counts, b2_stream_t stream);
/* mask[i] = (z[i] > thr_logit) ? 255 : 0 — the uint8 image of utils/pipeline.py:352-354 */
int b2_logits_to_mask(const float* z, int64_t count, float thr_logit, uint8_t* mask, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Optimizer step (utils/helpers.py:333-335): clip_grad_norm_(max_norm) + AdamW over all parameters in two launches.
 * `refs` is a DEVICE array of tensor references (fp32, element-wise aligned layouts); block b processes elements
 * [block_chunk[b]*chunk_elems, ...) of tensor block_tensor[b].  `step` (device float) is incremented by
 * b2_grad_sqnorm_multi and read by b2_adamw_multi for the bias correction; `lr` is a device float.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_tensor_ref {
  float* p;        /* parameter */
  const float* g;  /* gradient */
  float* m;        /* exp_avg */
  float* v;        /* exp_avg_sq */
  int64_t n;       /* elements */
} b2_tensor_ref;

int b2_grad_sqnorm_multi(const b2_tensor_ref* refs, const int32_t* block_tensor, const int32_t* block_chunk,
                         int32_t nblocks, int32_t chunk_elems, double* sqnorm, float* step, b2_stream_t stream);
int b2_adamw_multi(const b2_tensor_ref* refs, const int32_t* block_tensor, const int32_t* block_chunk,
                   int32_t nblocks, int32_t chunk_elems, const double* sqnorm, float max_norm, const float* lr,
                   float beta1, float beta2, float eps, float weight_decay, const float* step,
                   float* total_norm_out, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Multi-tensor weight re-pack (SURVEY.md §8f N1): one launch refreshes the bf16 MMA-layout copies (the outputs of
 * b2_pack_weights / b2_pack_weights_upfold / the im2col stem matrix) of EVERY convolution weight, right after
 * b2_adamw_multi updated the fp32 masters (utils/helpers.py:333-335), so that no conv call of the next step packs
 * anything.  `refs` is a DEVICE array; item_start = exclusive prefix sum of the per-tensor work items
 * (kind 0 / 1: ceil(cout/32) * ceil(cin/32) — one item is a 32 x 32 tile of all taps, ksize <= 3; kind 2:
 * ceil(cout/32) * ceil(cols/32));
 * total_items = their sum.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_pack_ref {
  const float* w;      /* fp32 [cout][cin][k][k] master, any strides */
  void* wf;            /* bf16 fprop layout (may be NULL) */
  void* wd;            /* bf16 dgrad layout (may be NULL) */
  int32_t cout, cin, ksize, kind;   /* kind: 0 plain, 1 UpConv-folded (ksize 3), 2 image-stem im2col matrix */
  int64_t s_co, s_ci, s_kh, s_kw;   /* element strides of w */
  int32_t item_start, pad_;         /* pad_: kind 2 -> columns of the stem matrix (multiple of 8) */
} b2_pack_ref;

int b2_pack_weights_multi(const b2_pack_ref* refs, int32_t nrefs, int32_t total_items, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * GPU input pipeline (SURVEY.md §8f N4): the reference's segmentation training transform (utils/trainer.py:88-101:
 * A.Resize(256,256) -> ShiftScaleRotate -> HorizontalFlip -> RandomBrightnessContrast -> Normalize -> ToTensorV2) and the
 * mask's / 255 (utils/dataset.py:124-126) in ONE kernel per batch: uint8 [N, Hs, Ws, 3] images + uint8 [N, Hs, Ws] masks
 * -> normalised fp32 NCHW [N, 3, S, S] + fp32 [N, 1, S, S], with the CPU pipeline's uint8 rounding points.  The random
 * draw stays on the host: `params` (DEVICE array, one entry per image) carries the inverse affine matrix in the resized
 * image's pixel coordinates, the flip flag and the brightness / contrast coefficients.  mean3 / std3 are HOST arrays.
 * Third-party arithmetic restated here: Albumentations 2.0.8 + OpenCV 4.12 (requirements.txt pins; neither is vendored
 * in the reference) — cv2.resize INTER_LINEAR (INTER_NEAREST for masks when mask_nearest_resize), cv2.warpAffine with
 * 1/32-pixel coordinate quantisation, BORDER_CONSTANT(0) or BORDER_REFLECT_101, the truncating uint8 LUT.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_aug_params {
  float m[6];            /* inverse affine: xs = m0*x + m1*y + m2, ys = m3*x + m4*y + m5 */
  float alpha, beta;     /* v' = clip(alpha * v + beta * 255) */
  int32_t flip, warp, adjust, border;   /* border: 0 constant(0), 1 reflect-101 */
} b2_aug_params;

int b2_seg_augment(const uint8_t* img, const uint8_t* mask, int32_t n, int32_t hs, int32_t ws, int32_t size,
                   const b2_aug_params* params, const float* mean3, const float* std3, int32_t mask_nearest_resize,
                   float* x, float* t, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * Attention gate, eval mode, ONE kernel (north_star (2); AttentionUNet.py:29-54 / R2AttU_Net.py:61-86 with the three
 * BatchNorms folded into weights, biases and two scalars):
 *     out = x * sigmoid(scale1 * (bpsi + wpsi . relu(W_g' g + W_x' x + bias')) + shift1)
 * runs as one tcgen05 GEMM with K = [g | x] (2C) and N = F_int whose epilogue reduces every accumulator row to psi
 * and writes x * psi — g1, x1, q and psi never touch HBM.  wpk = bf16 [1][fint][2C] = [s_g W_g | s_x W_x],
 * bias = s_g b_g + t_g + s_x b_x + t_x (fp32 [fint]); wpsi fp32 [fint]; bpsi / scale1 / shift1 device scalars.
 * Requires C % 64 == 0 and F_int in {32, 64, 128, 256}.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_gate_args {
  int32_t n, h, w, c, fint;
  const void* g;        /* NHWC bf16 [.., c] */
  int32_t ldg;
  const void* x;        /* NHWC bf16 [.., c] */
  int32_t ldx;
  const void* wpk;
  const float* bias;
  const float* wpsi;
  const float* bpsi;
  const float* scale1;
  const float* shift1;
  void* out;            /* NHWC bf16 [.., c] */
  int32_t ldo;
} b2_gate_args;

int b2_gate_fused(const b2_gate_args* args, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * ResNetUnet(freeze=False) (ResnetUnet.py:29-30: the torchvision ResNet-50 encoder trains too): what the encoder's
 * backward needs beyond the entry points above.
 *   b2_stem_im2col      the 7x7 / stride-2 / pad-3 stem (backbone.conv1) as a GEMM: fp32 NCHW image -> bf16 im2col
 *                       [N, Ho, Wo, cols] (column = tap * C + c, zero padded to `cols`), so that fprop (with the BN
 *                       statistics epilogue) and wgrad run on b2_conv_fprop / b2_conv_wgrad as a 1x1 convolution
 *   b2_maxpool3x3s2_bwd backward of backbone.maxpool = MaxPool2d(3, 2, 1): gather form, first maximum wins (ATen)
 *   b2_zero_insert2x    y[2h, 2w] = x[h, w], zero elsewhere: dY of a stride-2 convolution on the stride-1 grid — dgrad
 *                       and wgrad of the strided 3x3 / 1x1 convolutions then are the ordinary stride-1 kernels
 *   b2_relu_mask        g = out > 0 ? dy : 0, the gradient of relu(bn3(z) + identity) (torchvision Bottleneck)
 * ---------------------------------------------------------------------------------------------------------- */
int b2_stem_im2col(const float* x, int32_t n, int32_t c, int32_t h, int32_t w, int32_t ksize, int32_t stride,
                   int32_t pad, int32_t cols, void* xc, b2_stream_t stream);
int b2_maxpool3x3s2_bwd(const void* dy, int32_t lddy, const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w,
                        int32_t c, void* dx, int32_t lddx, b2_stream_t stream);
int b2_zero_insert2x(const void* x, int32_t ldx, int32_t n, int32_t h, int32_t w, int32_t c, void* y, int32_t ldy,
                     b2_stream_t stream);
int b2_relu_mask(const void* dy, int32_t lddy, const void* out, int32_t ldo, int64_t npix, int32_t c, void* g,
                 int32_t ldg, b2_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------
 * fp32 parity mode (BASELINE.json north_star: "fp32-accumulate mode within 1e-4"): the inference path with fp32
 * activation storage and fp32 FMA accumulation on the CUDA cores, for callers that need the reference's own fp32
 * results — utils/pipeline.py:340-357 runs `logits = model(img)` in fp32 without autocast and thresholds
 * sigmoid(logits) > 0.5.  Activations are NHWC fp32 [N, H, W, C] (channel stride ld*); weights are packed by
 * b2_f32_pack_weights to [tap][cin][cout] with the eval-mode BatchNorm folded in (W * scale[co], bias * scale + shift;
 * AttentionUNet.py:7-8 etc.).  b2_f32_conv covers every convolution of the four models: ksize <= 7, stride 1|2,
 * explicit padding, K from two tensors (elided torch.cat), + bias (+ addend before or after the ReLU), and the strided
 * output placement that turns ConvTranspose2d(k2, s2) (ResnetUnet.py:21,53) into four 1x1 convolutions.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct b2_f32_conv_args {
  const float* x0;        /* NHWC fp32 */
  const float* x1;        /* optional second K source */
  int32_t c0, c1, ldx0, ldx1;
  int32_t n, hi, wi;      /* input extent */
  int32_t ho, wo;         /* output grid extent (before out_mul) */
  int32_t ksize, stride, pad_h, pad_w;
  const float* w;         /* [ksize*ksize][c0 + c1][cout] */
  const float* bias;      /* [cout] or NULL */
  const float* addend;    /* optional NHWC fp32 [.., cout] on the OUTPUT grid (dense pixels, channel stride ldadd) */
  int32_t ldadd, add_after_act, relu, cout;
  float* y;               /* NHWC fp32 */
  int32_t ldy, out_mul, out_off_h, out_off_w;
} b2_f32_conv_args;

int b2_f32_conv(const b2_f32_conv_args* args, b2_stream_t stream);
int b2_f32_pack_weights(const float* w, int32_t cout, int32_t cin, int32_t ksize, int64_t s_co, int64_t s_ci,
                        int64_t s_kh, int64_t s_kw, const float* scale, const float* shift, const float* bias,
                        float* w_out, float* bias_out, b2_stream_t stream);
/* out = x * sigmoid(scale1 * (bpsi + wpsi . relu(g1 + x1)) + shift1): the attention gate after its two 1x1
 * convolutions (AttentionUNet.py:48-54); g1, x1 dense [npix][fint] */
int b2_f32_gate_tail(const float* g1, const float* x1, int32_t fint, const float* wpsi, const float* bpsi,
                     const float* scale1, const float* shift1, const float* x, int32_t ldx, int32_t c, int64_t npix,
                     float* out, int32_t ldo, b2_stream_t stream);
int b2_f32_maxpool(const float* x, int32_t n, int32_t h, int32_t w, int32_t c, int32_t ksize, int32_t stride,
                   int32_t pad, float* y, b2_stream_t stream);         /* nn.MaxPool2d(2,2) / (3,2,1) */
int b2_f32_upsample2x(const float* x, int32_t n, int32_t h, int32_t w, int32_t c, float* y, b2_stream_t stream);
int b2_f32_layout(const float* x, int32_t n, int32_t c, int64_t hw, int32_t to_nchw, float* y, b2_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200SEG_H_ */
