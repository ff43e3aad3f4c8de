/*
 * d3fk.h — C ABI of the B200-native (sm_100a) hot path for the d3f denoiser U-Net.
 *
 * The reference (ChainBreak/denoising_diffusion_deep_fake) has no FFI of its own: its hot path is
 * reached through a Python nn.Module call, `self.model(image_noisy)`
 * (d3f/train_denoiser/lit_module.py:117, d3f/train_deep_fake/lit_module.py:173,189,195,266), the
 * noising helper (train_denoiser/lit_module.py:128-153) and loss.backward().  Those calls bottom out
 * in ATen/cuDNN library ops; every entry point below replaces one family of those ops.  The Python
 * host (denoising_diffusion_deep_fake_b200/unet.py) builds a flat list of `d3fk_op` records once per
 * (batch, H, W, mode) and hands it to d3fk_run(); see INTEGRATION.md for the reference-side binding.
 *
 * Conventions: plain pointers and sizes only; the caller owns every buffer (activations, packed
 * weights, statistics, workspaces); nothing here allocates, synchronises or throws; all work is
 * enqueued on the given stream and is CUDA-graph-capture safe; return 0 or a negative D3FK_ERR_*.
 * There is no CPU path: on a device that is not sm_100 every launcher returns D3FK_ERR_ARCH.
 *
 * Tensors are NHWC ("pixel rows") inside the library: element (n,h,w,c) of a tensor with pixel
 * stride ld lives at ((n*H+h)*W+w)*ld + c.  dtype is D3FK_F32 (parity mode, CUDA-core FFMA
 * implicit GEMM) or D3FK_BF16 (tcgen05/TMEM implicit GEMM, fp32 accumulate).
 */
#ifndef D3FK_H
#define D3FK_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define D3FK_OK 0
#define D3FK_ERR_ARG (-1)
#define D3FK_ERR_ARCH (-2)
#define D3FK_ERR_CUDA (-3)
#define D3FK_ERR_UNSUPPORTED (-4)

#define D3FK_F32 0
#define D3FK_BF16 1

typedef void* d3fk_stream; /* cudaStream_t */

/* ---- convolution as implicit GEMM (replaces nn.Conv2d fwd and its dgrad; SURVEY §2.1 row 1) ----
 * mode 0: out[n,ho,wo,co] = sum_{kh,kw,c} A[n, ho*stride-pad+kh, wo*stride-pad+kw, c] * w[co][kh][kw][c]
 * mode 1 (transposed gather = dgrad of a conv with the same kh/kw/stride/pad):
 *         out[n,h,w,ci] = sum_{kh,kw,co} A[n,(h+pad-kh)/stride,(w+pad-kw)/stride,co] * w[ci][kh][kw][co]
 *         (terms whose coordinate is not divisible by stride or out of range are zero).
 * mode 2 (bf16 engine only; the 7x7 / stride-2 stem as a space-to-depth convolution): "windowed rows".  src0 is the
 *         space-to-depth image written by D3FK_OP_NCHW2S2D — [B][Hi][Wi + 3][ld0 = 16] with 2 zero pixels on the left and 1 on
 *         the right of every row — and the c0 = 64 "channels" of position (n, h, w) are the 64 CONTIGUOUS elements that start
 *         at padded pixel w, i.e. the 4-pixel window w-2 .. w+1 of the unpadded row: windows overlap, the pixel stride ld0 is
 *         smaller than c0.  out[n,ho,wo,co] = sum_{kh < 4, c < 64} src0[n, ho - pad + kh, window wo][c] * w[co][kh][c]
 *         (kw = 1, stride 1, pad = 2 in h only, Ho = Hi, Wo = Wi; weights from D3FK_OP_PACK_STEM).  Each (pixel, kh) is one
 *         128-byte operand row, so the whole A tile is a TMA box: K = 256 (4 k-blocks, none of them padding) instead of the
 *         392 of the 7x7 gather, and no per-thread gather.
 * A is the channel concatenation of src0 (c0 channels, optionally read through a nearest 2x upsample:
 * F.interpolate(scale_factor=2) + torch.cat of smp's DecoderBlock) and src1 (c1 channels).
 * Epilogue: v = acc; v = v*scale[c]+shift[c] (if scale); v += res (if res); v = max(v,0) (if relu);
 * stats[c] += v, stats[Cout+c] += v*v (if stats; per-channel batch statistics for train-mode BN);
 * store to `out` (NHWC dtype) or, if out_nchw is set, to fp32 NCHW (the U-Net's output tensor). */
typedef struct d3fk_conv_params {
  int32_t dtype, mode;
  const void* src0; const void* src1;
  int32_t c0, c1, ld0, ld1, up0;
  int32_t B, Hi, Wi, Ho, Wo;
  int32_t kh, kw, stride, pad;
  const void* w; int32_t Cout, _pad0;
  void* out; float* out_nchw;
  const float* scale; const float* shift;
  const void* res;
  double* stats;
  int32_t ldo, ldr, relu, _pad1;
  void* ws; int64_t ws_bytes;   /* unused since split K reduces inside a thread-block cluster (kept for ABI stability) */
  /* BN-backward reduction fused into a dgrad epilogue (bw_x != NULL; bf16 engine): the output is the gradient g wrt the
   * activation of a conv -> BN -> ReLU layer whose raw conv output is bw_x (pixel stride bw_ldx), activation bw_act and saved
   * statistics bw_mean / bw_invstd; `stats` then receives sum(g') and sum(g' * xhat), g' = g where bw_act > 0 (if bw_relu)
   * else 0, xhat = (bw_x - mean) * invstd — the two sums of d3fk_bn_bwd_reduce, without its pass over g, x and act. */
  const void* bw_x; const void* bw_act; const float* bw_mean; const float* bw_invstd;
  int32_t bw_ldx, bw_ldact, bw_relu, _pad2;
} d3fk_conv_params;

/* ---- weight gradient (replaces cuDNN wgrad): dw[co][ci][kh][kw] += sum_{n,ho,wo} dy[n,ho,wo,co] * A[...]
 * with the same mode-0 gather as the forward conv.  dw is the fp32 OIHW master-gradient tensor
 * (cin_real input channels); contributions are added with atomics, the caller zeroes it first.  cin_real is the extent
 * (= stride) of dw's input-channel dimension: a launch over a channel sub-range of the input (c0 + c1 < cin_real, src0 and
 * dw offset to the first channel of the range) accumulates that slice of dw. */
typedef struct d3fk_wgrad_params {
  int32_t dtype;
  int32_t mode;   /* 0: the gather above.  2 (bf16 engine): the space-to-depth stem, operands as conv mode 2 (src0 = the padded
                     space-to-depth image, c0 = 64 window channels, ld0 = 16, kh = 4, kw = 1, pad = 2); dw is still the 7x7 OIHW
                     master gradient (cin_real = 3): row k = th*64 + tw*16 + (dy*2+dx)*4 + ci lands on tap (2th+dy-1, 2tw+dx-1) */
  const void* src0; const void* src1;
  int32_t c0, c1, ld0, ld1, up0;
  int32_t B, Hi, Wi, Ho, Wo;
  int32_t kh, kw, stride, pad;
  const void* dy; float* dw;
  int32_t ldy, Cout, cin_real, cout_real;
} d3fk_wgrad_params;

/* ---- grouped weight gradient: `count` problems of IDENTICAL geometry (the 3x3 / stride-1 convolutions of one ResNet stage)
 * in ONE launch.  `base` describes the geometry (its src0 / dy / dw are ignored); problem i reads src0[i], dy[i] and writes
 * dw[i].  Single-source layers only (base.c1 == 0).  The deep stages' weight gradients are tiny GEMMs (4096 or 1024 pixels
 * of reduction): launched one by one each needs a pixel split over a cluster, a reduction and ~20 us of fixed cost; grouped,
 * the output tiles of the whole stage fill the chip and each CTA reduces over all (or most) pixels. */
#define D3FK_WGRAD_GROUP_MAX 12
typedef struct d3fk_wgrad_group_params {
  d3fk_wgrad_params base;
  int32_t count, _pad0;
  const void* src0[D3FK_WGRAD_GROUP_MAX];
  const void* dy[D3FK_WGRAD_GROUP_MAX];
  float* dw[D3FK_WGRAD_GROUP_MAX];
} d3fk_wgrad_group_params;

/* ---- weight packing: fp32 OIHW master -> [Cout][kh][kw][cin_pad] (forward) and/or
 * [Cin][kh][kw][cout_pad] (dgrad) in dtype, zero padded. */
typedef struct d3fk_pack_params {
  int32_t dtype, Cout, Cin, kh, kw, cin_pad, cout_pad, blk0;   /* blk0: PACK_ALL only — first 32x32 block of this layer */
  const float* w; void* w_fwd; void* w_dgrad;
} d3fk_pack_params;

/* ---- BatchNorm2d (+residual) + ReLU, train and eval, forward and backward
 * (replaces nn.BatchNorm2d / ReLU / BasicBlock `out += identity`; SURVEY §2.1 rows 2-4).
 * bn_apply with `stats` set finalises the batch statistics itself (mean/invstd/running stats written by block 0)
 * and ignores scale/shift; with stats == NULL it applies the given scale/shift.  bn_bwd_apply derives its
 * coefficients from bstats/mean/invstd/gamma and writes dgamma/dbeta; bn_finalize / bn_bwd_finalize remain as
 * stand-alone entry points.  bn_fold with mean / invstd set also writes running_mean and 1/sqrt(running_var + eps) there (the
 * rows a frozen backward reads). */
typedef struct d3fk_bn_params {
  int32_t dtype, C, relu;
  int32_t mask_from_x;                  /* backward: ReLU mask = (x*scale + shift > 0) instead of reading `act` — valid when the
                                           forward had no residual (train forward publishes scale / shift for this) */
  int64_t count;                        /* B*H*W */
  const void* x; void* y; const void* res;
  int32_t ldx, ldy, ldr;
  int32_t frozen;                       /* backward on the running statistics (eval-mode BN: mean / invstd hold the running values
                                           BN_FOLD wrote): dx = gamma*invstd*dy', no term from the reductions; dgamma / dbeta as usual */
  double* stats;                        /* [2][C] sum, sumsq of x (from the conv epilogue) */
  const float* gamma; const float* beta;
  float* running_mean; float* running_var; int64_t* num_batches_tracked;
  float eps, momentum;
  float* scale; float* shift;           /* y = x*scale + shift */
  float* mean; float* invstd;
  /* backward */
  const void* dy; const void* act;      /* grad wrt y; y itself (ReLU mask = act > 0) */
  void* dx; void* dres;                 /* grad wrt x; masked grad for the residual branch (nullable) */
  int32_t lddy, ldact, lddx, lddres;
  double* bstats;                       /* [2][C] sum dy', sum dy'*xhat */
  float* dgamma; float* dbeta;
  float* coef;                          /* [3][C] scratch written by bn_bwd_finalize (nullable) */
  uint32_t* barrier;                    /* D3FK_OP_BN_BWD: zeroed grid-barrier counter (NULL: reduce and apply as two kernels) */
} d3fk_bn_params;

/* ---- convolution + train-mode BatchNorm (+residual) + ReLU as ONE op (the forward of every conv->BN->ReLU of the U-Net).
 * Semantics = d3fk_conv(conv) followed by d3fk_bn_apply(bn) with bn.x == conv.out and bn.stats == conv.stats.  When every
 * output tile of the layer is resident at once the library fuses the two: the conv kernel finalises the statistics behind a
 * grid-wide barrier (`barrier`: a zeroed uint32 the caller clears with the statistics) and writes raw output and activation
 * itself.  barrier == NULL forces the two-kernel form. */
typedef struct d3fk_convbn_params {
  d3fk_conv_params conv;
  d3fk_bn_params bn;
  uint32_t* barrier;
} d3fk_convbn_params;

/* ---- MaxPool2d(3,2,1) fwd/bwd, 2x2 sum pool (= backward of nearest 2x upsample), NCHW fp32 -> NHWC */
typedef struct d3fk_pool_params {
  int32_t dtype, B, H, W, C, accumulate;  /* H,W: input extent of the forward op */
  const void* x; void* y; uint8_t* idx;
  const void* dy; void* dx;
  int32_t ldx, ldy, lddy, lddx;
} d3fk_pool_params;

typedef struct d3fk_layout_params {
  int32_t dtype, B, C, H, W, cpad;
  const float* src; void* dst;            /* src fp32 NCHW [B,C,H,W] -> dst NHWC dtype [B,H,W,cpad] */
  float* chansum;                         /* D3FK_OP_NCHW2NHWC, nullable, C <= 8: chansum[c] += sum over pixels of the (dtype-rounded) values
                                             written — the bias gradient of the head, without a second pass over dst */
} d3fk_layout_params;

/* nearest 2x upsample of src0 + channel concat with src1, materialised (smp DecoderBlock: F.interpolate(scale_factor=2) +
 * torch.cat): out[n,h,w, 0:c0] = src0[n, h/2, w/2, :], out[n,h,w, c0:c0+c1] = src1[n,h,w,:].  H, W = OUTPUT extent.  Used
 * for the decoder convolutions that then run on the slab path (one HBM pass instead of a 9x gather). */
typedef struct d3fk_upcat_params {
  int32_t dtype, B, H, W, c0, c1, ld0, ld1, ldo, _pad0;
  const void* src0; const void* src1; void* out;
} d3fk_upcat_params;

/* ---- video-frame pre / post-processing, batched (SURVEY §8 row f4).
 * frames_to_tensor replaces LitModule.cv2_to_tensor_normalised (d3f/train_deep_fake/lit_module.py:272-283):
 *   uint8 BGR HWC [N,H,W,3] -> fp32 RGB NCHW [N,3,H,W],  t = (float(v) - mean_c*255) / (std_c*255)   (two fp32 roundings)
 * tensor_to_frames replaces LitModule.tensor_cv2_to_denormalised (:285-300):
 *   fp32 RGB NCHW -> uint8 BGR HWC,  v = clamp(int(t*(std_c*255) + mean_c*255), 0, 255)  (product and sum rounded
 *   separately, conversion truncates toward zero as tensor.int() does and saturates beyond int32 as it does on a CUDA
 *   device).  mean / std are in RGB order (the configs' order).
 * `frames` is read by to_tensor and written by to_frames; `tensor` the other way round. */
typedef struct d3fk_frames_params {
  int32_t N, H, W, _pad0;
  uint8_t* frames; float* tensor;
  float mean[3], std[3];
} d3fk_frames_params;

/* per-channel sum over (n,h,w) of an NHWC tensor into fp32 out[c] (head bias gradient) */
typedef struct d3fk_chansum_params {
  int32_t dtype, C, ld, _pad0; int64_t count;
  const void* x; float* out;
} d3fk_chansum_params;

/* ---- noising q_sample (d3f/train_denoiser/lit_module.py:128-153) -------------------------------
 * r_b = 1/lam * log(1/(y_b*(1-c)+c)), c = e^-lam;  out = sqrt(1-r_b)*x + sqrt(r_b)*noise.
 * noise / y may be supplied (parity runs) or drawn in-kernel from Philox4x32-10(seed, offset).
 * fixed_r >= 0 overrides the draw (balance_training_images/lit_module.py:109-120 uses 0.7). */
typedef struct d3fk_qsample_params {
  int32_t B, chw; float lam, fixed_r;
  const float* x; const float* noise; const float* y;
  float* out; float* r_out; float* noise_out;
  uint64_t seed, offset;
} d3fk_qsample_params;

/* ---- random affine augmentation fused with the noising (SURVEY §8 row f3).  Replaces
 * `image = self.shared_augmentation_sequence(image)` (kornia RandomAffine, d3f/train_denoiser/lit_module.py:55-65, :113)
 * followed by blend_random_amount_of_noise_with_each_sample (:115): one pass reads x and writes BOTH the augmented clean
 * image (the loss target) and its noised version.
 * minv: B x 6 floats, the INVERSE map of each sample, output pixel (ox, oy) -> source pixel
 *   sx = m0*ox + m1*oy + m2,  sy = m3*ox + m4*oy + m5     (pixel centres at integer coordinates)
 * sampled bilinearly with zero padding outside the image.  Noise / ratio exactly as d3fk_q_sample applied to the augmented
 * image (same Philox counters), so affine_q_sample(x) == q_sample(affine(x)) bit for bit. */
typedef struct d3fk_affine_qsample_params {
  int32_t B, C, H, W; float lam, fixed_r;
  const float* x; const float* minv; const float* noise; const float* y;
  float* out_aug; float* out_noisy; float* r_out;
  uint64_t seed, offset;
} d3fk_affine_qsample_params;

/* ---- posterior update x_{i-1} = k_xi*x_i + k_x0*x0_hat + sigma*z (SURVEY §8a row S) ------------
 * Coefficients come from coef_table[*step][0..3] = (k_xi, k_x0, sigma, r_prev) when coef_table is set (CUDA-graph
 * replay: the graph is step-independent), else from the immediates. z supplied or Philox(seed, offset+*step): counter
 * (i, i >> 32, off, off >> 32) for the 4-element vector i of the op's (sub-)batch.
 * Masked form (mask != NULL; replacement inpainting): x is NCHW with chw = C*H*W elements per sample and hw = H*W, src
 * has x's shape and mask is [B][H][W] (broadcast over channels, clamped to [0, 1]; 1 = generate, 0 = keep):
 *   known = sqrt(1 - r_prev)*src + sqrt(r_prev)*n      (rounded as d3fk_q_sample with fixed_r = r_prev: known == src at 0)
 *   x     = m*post + (1 - m)*known                      (fma(m, post, (1 - m)*known): exactly post at m = 1, known at 0)
 * n is known_noise when supplied, else drawn in-kernel from a stream no other draw uses: the key and offset of z with
 * bit 31 set in counter word 1, i.e. counter (i, (i >> 32) | 0x80000000, off, off >> 32).  z is the unmasked kernel's, so
 * a mask of ones reproduces the unmasked update bit for bit.  x0_hat may alias x. */
typedef struct d3fk_posterior_params {
  int64_t n;
  float* x; const float* x0_hat; const float* z;
  const float* coef_table; const int32_t* step;
  float k_xi, k_x0, sigma, r_prev;
  uint64_t seed, offset;
  const float* src; const float* mask; const float* known_noise;   /* masked form: all NULL for the plain update */
  int32_t chw, hw;
} d3fk_posterior_params;

/* ---- second-order multistep update (DPM-Solver++ 2M in data-prediction form; k-diffusion's dpmpp_2m at eta = 0 and
 * dpmpp_2m_sde, midpoint, at eta > 0), in the variance-preserving ratio r: lambda(r) = ln((1 - r)/r)/2 (-inf at r = 1,
 * +inf at 0), alpha = sqrt(1 - r), s = sqrt(r).  Step i goes from r_i to r_t with h_i = lambda(r_t) - lambda(r_i):
 *   D_i     = x0_i + c_i*(x0_i - x0_{i-1})                       (x0_{i-1}: the previous step's x0_hat, kept in x0_prev)
 *   x_{i+1} = k_xi*x_i + k_x0*D_i + sigma*z
 *   k_xi = (s_t/s_i) e^{-eta h},  k_x0 = alpha_t (1 - e^{-(1+eta) h}),  sigma = s_t sqrt(1 - e^{-2 eta h}),
 *   c_i  = h_i / (2 h_{i-1})
 * c_i = 0 on the first step and wherever h_i or h_{i-1} is infinite; a step to r_t = 0 is (0, 1, 0, 0, 0) and returns
 * x0_hat.  At eta = 0 and eta = 1 (k_xi, k_x0, sigma) equal the first-order posterior's, so a row with c = 0 is today's
 * update.  Rounding: d = h - p, D = fma(c, d, h), then the posterior's (fma(k_xi, x, k_x0*D), fma(sigma, z, .)): with
 * c = 0 the result is bit-identical to d3fk_posterior_step with the same coefficients, and x0_prev is not read.
 * Every vector whose update is computed copies x0_hat into x0_prev (the masked form skips all-0 mask vectors, which
 * read no x0_hat either).  z and the masked known noise are the posterior's streams.  Table form: base.coef_table rows
 * are 5 floats (k_xi, k_x0, sigma, r_prev, c) indexed by *base.step.  x0_hat may alias x, never x0_prev. */
typedef struct d3fk_posterior_2m_params {
  d3fk_posterior_params base;
  float* x0_prev; float c; int32_t _pad;
} d3fk_posterior_2m_params;   /* 128 bytes */

typedef struct d3fk_misc_params {          /* MEMSET: p0[0..n) bytes = 0; INC: *(int32*)p0 += 1; PACK_ALL: see enum */
  void* p0; int64_t n;
} d3fk_misc_params;

/* ---- fused Adam (+EMA lerp) over a flat fp32 arena (torch.optim.Adam semantics: eps outside sqrt,
 * no weight decay, no amsgrad; d3f/train_denoiser/lit_module.py:95, train_deep_fake/lit_module.py:116-120).
 * bias1 = 1 - beta1^step, bias2 = 1 - beta2^step (the caller's step count). */
typedef struct d3fk_adam_params {
  int64_t n;
  float* p; const float* g; float* m; float* v; float* ema;
  float lr, beta1, beta2, eps, bias1, bias2, ema_decay, grad_scale;
  const float* dyn;   /* nullable: device floats {lr, bias1, bias2, ema_decay} that override the immediates — the per-step
                         scalars of a launch recorded once in a CUDA graph and replayed every training step */
} d3fk_adam_params;

/* ---- four floats written to device memory by value (no host buffer to race with): the per-step scalars `dyn` of the
 * Adam launches inside a replayed CUDA graph are refreshed with this launch in front of every replay. */
typedef struct d3fk_scalars_params {
  float* dst; float v[4];
} d3fk_scalars_params;

/* ---- fused MSE + (1 - SSIM) criterion, forward and gradient
 * (d3f/loss_functions/structural_similarity_loss.py:14-26 + piqa.SSIM defaults, SURVEY Appendix B1).
 * acc[0] += sum (pred-target)^2 ; acc[1] += sum of the SSIM map; the caller zeroes acc and forms
 * loss = (acc[0]/numel + 1 - acc[1]/(B*C*(H-10)*(W-10))) / 2.  grad (nullable) receives grad_scale * dL/dpred, with
 * torch's clip(0, 1) subgradient on the normalised prediction: the SSIM term passes where lo <= pred <= hi (both ends
 * included) and is zero strictly outside; the MSE term passes everywhere. */
typedef struct d3fk_loss_params {
  int32_t B, C, H, W;
  const float* pred; const float* target;   /* fp32 NCHW */
  float* grad; double* acc;
  float lo, hi, grad_scale, _pad0;
  float win[12];                             /* 11-tap normalised Gaussian (+1 pad) */
  float* loss_out;                           /* nullable.  When set, acc must hold 3 zeroed doubles: the last block writes the
                                                finished scalar loss here and re-zeroes acc (self-resetting workspace) */
} d3fk_loss_params;

enum d3fk_op_kind {
  D3FK_OP_CONV = 1, D3FK_OP_WGRAD = 2, D3FK_OP_PACK = 3, D3FK_OP_NCHW2NHWC = 4,
  D3FK_OP_BN_FINALIZE = 5, D3FK_OP_BN_APPLY = 6, D3FK_OP_BN_FOLD = 7,
  D3FK_OP_BN_BWD_REDUCE = 8, D3FK_OP_BN_BWD_FINALIZE = 9, D3FK_OP_BN_BWD_APPLY = 10,
  D3FK_OP_MAXPOOL_FWD = 11, D3FK_OP_MAXPOOL_BWD = 12, D3FK_OP_SUMPOOL2 = 13,
  D3FK_OP_CHANSUM = 14, D3FK_OP_QSAMPLE = 15, D3FK_OP_POSTERIOR = 16,
  D3FK_OP_MEMSET = 17, D3FK_OP_INC = 18, D3FK_OP_ADAM = 19,
  D3FK_OP_PACK_ALL = 20, /* misc: p0 = device array of d3fk_pack_params, n = (blocks << 17) | (count << 1) | is_bf16 */
  D3FK_OP_LOSS = 21,
  D3FK_OP_CONV_BN = 22,
  D3FK_OP_UPCAT = 23,
  D3FK_OP_FRAMES_TO_TENSOR = 26, D3FK_OP_TENSOR_TO_FRAMES = 27,   /* frames params */
  D3FK_OP_AFFINE_QSAMPLE = 28,
  D3FK_OP_SET_SCALARS = 29,   /* scalars params */
  D3FK_OP_JOIN = 30,          /* misc params: n = lane to join back into the main stream */
  D3FK_OP_WGRAD_GROUP = 25,   /* wgrad_group params; forked onto the side streams like D3FK_OP_WGRAD */
  D3FK_OP_BN_BWD = 24,   /* bn params: bn_bwd_reduce + bn_bwd_apply as one op (one kernel behind a grid barrier when `barrier` is set).
                            frozen: ONE streaming pass writes dx (and dres) and accumulates bstats, then bn_bwd_finalize writes dgamma / dbeta */
  D3FK_OP_NCHW2S2D = 31,   /* layout params (C = 3, cpad = 4, H and W even): fp32 NCHW -> the padded space-to-depth image of conv mode 2:
                              dst[b][h/2][w/2 + 2][((h%2)*2 + (w%2))*4 + c]; the pad pixels / channel are left untouched (zero them once) */
  D3FK_OP_PACK_STEM = 32,  /* pack params (Cout, Cin = 3, kh = kw = 7): w_fwd[co][th*64 + tw*16 + (dy*2+dx)*4 + ci] =
                              w[co][ci][2*th+dy-1][2*tw+dx-1] (0 outside the 7x7 window and for ci = 3): the conv mode 2 weights */
  D3FK_OP_POSTERIOR_2M = 33   /* posterior_2m params: the second-order multistep update (5-float table rows) */
};

/* `lane`: 0 = the caller's stream (the main chain).  lane 1..D3FK_MAX_LANES = an internal branch stream: the op runs there,
 * ordered behind everything the main stream held when the branch's first op was reached (fork), and the main stream picks
 * the branch up again at D3FK_OP_JOIN (misc.n = lane; any lane still open at the end of the list is joined there).  Used
 * for the 1x1 / stride-2 downsample branch of a ResNet stage's first block, which is independent of the block's conv1 ->
 * BN -> ReLU chain until the residual add (torchvision BasicBlock.forward, resnet.py:89-105).  Branch ops never wait on a
 * grid-wide barrier (the plans emit their two-kernel forms), so two co-scheduled kernels cannot deadlock on residency. */
#define D3FK_MAX_LANES 2
typedef struct d3fk_op {
  int32_t kind, lane;
  union {
    d3fk_conv_params conv; d3fk_wgrad_params wgrad; d3fk_pack_params pack; d3fk_bn_params bn;
    d3fk_pool_params pool; d3fk_layout_params layout; d3fk_chansum_params chansum;
    d3fk_qsample_params qsample; d3fk_posterior_params posterior; d3fk_misc_params misc;
    d3fk_adam_params adam; d3fk_loss_params loss; d3fk_convbn_params convbn; d3fk_upcat_params upcat;
    d3fk_wgrad_group_params wgrad_group; d3fk_frames_params frames; d3fk_affine_qsample_params affine_qsample;
    d3fk_scalars_params scalars; d3fk_posterior_2m_params posterior_2m;
  } u;
} d3fk_op;

/* library / device */
int d3fk_version(void);
int d3fk_sizeof_op(void);                 /* ABI check for the host-side struct mirror */
int d3fk_init(int device);                /* D3FK_ERR_ARCH unless the device is sm_100 */
const char* d3fk_last_error(void);
int d3fk_device_error_flag(void);         /* non-zero if a kernel hit its barrier watchdog (debug) */
int d3fk_debug_timeline(unsigned long long* out, int n, unsigned* launches);   /* phase stamps of -DD3FK_TIMELINE builds */

/* run a recorded op list on `stream` (the hot path: one call per U-Net forward / backward) */
int d3fk_run(const d3fk_op* ops, int n_ops, d3fk_stream stream);

/* Weight-gradient ops (D3FK_OP_WGRAD) of a list are forked onto an internal side stream (they are off the backward
 * critical path); d3fk_run joins that stream back into `stream` before it returns to the caller.  d3fk_run_nojoin leaves
 * the side stream running — backward segments can then overlap the weight gradients of earlier segments — and the caller
 * joins ONCE with d3fk_side_stream_join(stream) before anything reads the weight gradients (optimizer, allreduce). */
int d3fk_run_nojoin(const d3fk_op* ops, int n_ops, d3fk_stream stream);
int d3fk_side_stream_join(d3fk_stream stream);

/* profiling aid: as d3fk_run, but brackets every op with CUDA events and returns per-op milliseconds
 * (synchronises the stream; allocates events — never used on the hot path) */
int d3fk_run_profile(const d3fk_op* ops, int n_ops, d3fk_stream stream, float* ms_per_op);

/* single-op entry points (same launchers; used by the per-op parity tests) */
int d3fk_conv(const d3fk_conv_params* p, d3fk_stream stream);
int d3fk_wgrad(const d3fk_wgrad_params* p, d3fk_stream stream);
int d3fk_wgrad_group(const d3fk_wgrad_group_params* p, d3fk_stream stream);
int d3fk_frames_to_tensor(const d3fk_frames_params* p, d3fk_stream stream);
int d3fk_tensor_to_frames(const d3fk_frames_params* p, d3fk_stream stream);
int d3fk_affine_q_sample(const d3fk_affine_qsample_params* p, d3fk_stream stream);
int d3fk_conv_bn(const d3fk_convbn_params* p, d3fk_stream stream);
int d3fk_pack_weights(const d3fk_pack_params* p, d3fk_stream stream);
int d3fk_nchw_to_nhwc(const d3fk_layout_params* p, d3fk_stream stream);
int d3fk_bn_finalize(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_apply(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_fold(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_bwd_reduce(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_bwd_finalize(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_bwd_apply(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_bn_bwd(const d3fk_bn_params* p, d3fk_stream stream);
int d3fk_maxpool_fwd(const d3fk_pool_params* p, d3fk_stream stream);
int d3fk_maxpool_bwd(const d3fk_pool_params* p, d3fk_stream stream);
int d3fk_sumpool2(const d3fk_pool_params* p, d3fk_stream stream);
int d3fk_chansum(const d3fk_chansum_params* p, d3fk_stream stream);
int d3fk_upcat(const d3fk_upcat_params* p, d3fk_stream stream);
int d3fk_q_sample(const d3fk_qsample_params* p, d3fk_stream stream);
int d3fk_posterior_step(const d3fk_posterior_params* p, d3fk_stream stream);
int d3fk_posterior_2m_step(const d3fk_posterior_2m_params* p, d3fk_stream stream);
int d3fk_adam(const d3fk_adam_params* p, d3fk_stream stream);
int d3fk_set_scalars(const d3fk_scalars_params* p, d3fk_stream stream);
int d3fk_mse_ssim_loss(const d3fk_loss_params* p, d3fk_stream stream);

/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t d3fk_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif
