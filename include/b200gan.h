/*
 * b200gan.h -- C ABI of libb200gan.so: the sm_100a implementation of the
 * Generator/Discriminator hot path of eriklindernoren/PyTorch-GAN.
 *
 * The reference has no FFI of its own: its operator boundary is the torch.nn.Module
 * protocol (SURVEY.md section 8b).  Each entry point below replaces the arithmetic that one
 * reference call site hands to third-party torch; the reference file:line is cited per
 * function.  All signatures are plain C: raw device pointers, sizes, a cudaStream_t passed
 * as void*.  No torch types cross this boundary.
 *
 * Conventions
 *   - Activations are fp32, NHWC ("channels_last"), dense: x[n][h][w][c].
 *   - Weight parameters stay in PyTorch's external layout (Conv2d: OIHW, ConvTranspose2d:
 *     IOHW) so state_dict keys/shapes are unchanged (pix2pix.py:71-72, cyclegan.py:75-78);
 *     packed copies are derived caches produced by b200gan_pack_weights().
 *   - Every launch is asynchronous on the given stream; nothing allocates or frees device
 *     memory; nothing synchronises the host.  All buffers are caller-owned.
 *   - Return value: 0 = OK, negative = B200GAN_E_*; b200gan_last_error() gives the text
 *     (thread-local).  There is no CPU fallback anywhere in this library.
 */
#ifndef B200GAN_H
#define B200GAN_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GAN_VERSION 100

enum {
  B200GAN_OK = 0,
  B200GAN_E_UNSUPPORTED = -1, /* geometry not supported by the requested algorithm */
  B200GAN_E_BAD_ARG = -2,     /* null pointer, misalignment, inconsistent sizes */
  B200GAN_E_CUDA = -3,        /* a CUDA runtime/driver call failed */
  B200GAN_E_ARCH = -4         /* device is not sm_100 */
};

/* activation fused into an epilogue / applied by a norm kernel */
enum { B200GAN_ACT_NONE = 0, B200GAN_ACT_LRELU = 1, B200GAN_ACT_RELU = 2, B200GAN_ACT_TANH = 3,
       B200GAN_ACT_SIGMOID = 4 };

/* algorithm selector for the convolution entry points */
enum { B200GAN_ALGO_AUTO = 0, /* tcgen05 when the geometry qualifies, else SIMT */
       B200GAN_ALGO_SIMT = 1, /* fp32 FFMA implicit GEMM (any geometry) */
       B200GAN_ALGO_TC = 2 }; /* tcgen05 TF32 implicit GEMM (error if unsupported) */

/* padding mode of the (virtual) padded input */
enum { B200GAN_PAD_ZERO = 0, B200GAN_PAD_REFLECT = 1 };

/* packed-weight layouts produced by b200gan_pack_weights() */
enum {
  B200GAN_PACK_SIMT_FPROP = 0, /* [R][S][Cin][Cout]   : conv fprop / convT dgrad, SIMT        */
  B200GAN_PACK_SIMT_DGRAD = 1, /* [R][S][Cout][Cin]   : conv dgrad / convT fprop, SIMT        */
  B200GAN_PACK_TC_FPROP = 2,   /* [R*S][Cout][Cin]    tf32-rounded, K-major, tcgen05 fprop    */
  B200GAN_PACK_TC_DGRAD = 3,   /* [R*S][Cin][Cout]    tf32-rounded, taps flipped, dgrad       */
  B200GAN_PACK_TC_FPROP_UP2 = 4, /* [4 phases][4 taps][Cout][Cin]: 3x3 s1 p1 conv folded with a
                                    preceding nearest x2 upsample into four 2x2 phase filters  */
  B200GAN_PACK_TC_DGRAD_UP2 = 5  /* [4 phases][4 taps][Cin][Cout]: its data gradient           */
};

/*
 * Geometry of one convolution call site.  Replaces the constructor arguments of
 *   nn.Conv2d           dcgan.py:55,59,62,78  pix2pix/models.py:23,79,115,127
 *                       cyclegan/models.py:28,32,50,60,75,82,106,118
 *   nn.ConvTranspose2d  pix2pix/models.py:39
 * optionally composed with the shape-only modules the reference places directly in front:
 *   nn.Upsample(scale_factor=2)   dcgan.py:54,58  cyclegan/models.py:74  pix2pix/models.py:77
 *   nn.ZeroPad2d((1,0,1,0))       pix2pix/models.py:78,126   cyclegan/models.py:117
 *   nn.ReflectionPad2d(k)         cyclegan/models.py:27,31,49,81
 * The "virtual input" is  pad(upsample(x)): size (H*up + pad_t + pad_b) x (W*up + pad_l + pad_r).
 */
typedef struct b200gan_conv_geom {
  int32_t N, H, W, C;  /* stored input tensor (before upsample / padding), NHWC          */
  int32_t K;           /* output channels                                                  */
  int32_t R, S;        /* filter height, width                                             */
  int32_t stride;      /* same in h and w                                                  */
  int32_t pad_t, pad_l, pad_b, pad_r; /* total padding of the virtual input (conv padding +
                                         any folded ZeroPad2d / ReflectionPad2d)           */
  int32_t pad_mode;    /* B200GAN_PAD_*                                                    */
  int32_t up;          /* 1, or 2 = nearest-neighbour x2 upsample folded in front          */
  int32_t transposed;  /* 0 = Conv2d, 1 = ConvTranspose2d (pad_* = its `padding`, up == 1) */
  int32_t P, Q;        /* output height, width (checked against the other fields)          */
} b200gan_conv_geom;

/* Epilogue fused into fprop:  y = chan_scale[n,k] * act(conv + bias[k])  (each part optional).
 * stats (optional) receives, atomically accumulated in fp64, the per-group sums of y and y*y
 * that the following BatchNorm2d / InstanceNorm2d needs: stats[0..G) = sum, stats[G..2G) =
 * sum of squares, G = K (stats_per_sample == 0) or N*K (== 1).  Caller zeroes it. */
typedef struct b200gan_epilogue {
  const float *bias;       /* [K] or NULL                                                  */
  int32_t act;             /* B200GAN_ACT_*                                                */
  float slope;             /* LeakyReLU negative slope                                     */
  const float *chan_scale; /* [N][K] Dropout2d keep-mask / (1-p)  (dcgan.py:77) or NULL    */
  double *stats;           /* [2][G] or NULL                                               */
  int32_t stats_per_sample;
  int32_t round_tf32;      /* store y rounded to TF32 (RN) so that a following tcgen05 conv
                              consumes exactly-representable operands                      */
} b200gan_epilogue;

int b200gan_version(void);
const char *b200gan_last_error(void);
/* 0 if the current device is sm_100 and the tcgen05/TMA paths can run, else B200GAN_E_ARCH */
int b200gan_check_device(void);

/* ---- weights ------------------------------------------------------------------------ */
size_t b200gan_packed_weight_floats(const b200gan_conv_geom *g, int pack);
/* w: the nn.Parameter storage (Conv2d [K][C][R][S]; ConvTranspose2d [C][K][R][S]). */
int b200gan_pack_weights(const b200gan_conv_geom *g, int pack, const float *w, float *packed,
                         void *stream);

/* Every packed copy of an optimizer's weights in ONE launch (the job table travels as a kernel argument): called by
 * b200gan.optim.Adam right after the parameter update, so a training step carries 2 pack launches instead of ~20. */
typedef struct b200gan_pack_job {
  const float *w;
  float *packed;
  b200gan_conv_geom geom;
  int32_t pack; /* B200GAN_PACK_* */
} b200gan_pack_job;
int b200gan_pack_weights_multi(const b200gan_pack_job *jobs, int32_t count, void *stream);

/* ---- convolution: forward, data gradient, weight gradient ---------------------------- */
/* 1 if algo (B200GAN_ALGO_TC) supports this geometry for the given pass (0 fprop,1 dgrad,2 wgrad) */
int b200gan_conv2d_supported(const b200gan_conv_geom *g, int pass, int algo);

/* y[N][P][Q][K] = epilogue(conv(x, w)).  `packed` must be the layout the algorithm wants:
 * SIMT: PACK_SIMT_FPROP (Conv2d) / PACK_SIMT_DGRAD (ConvTranspose2d);
 * TC  : PACK_TC_FPROP, or PACK_TC_FPROP_UP2 when g->up == 2.
 * Replaces cudnnConvolutionForward behind nn.Conv2d.forward (dcgan.py:69,95). */
int b200gan_conv2d_fprop(const b200gan_conv_geom *g, const b200gan_epilogue *ep, const float *x,
                         const float *packed, float *y, int algo, void *stream);

/* dx[N][H][W][C] = d(loss)/dx given dy[N][P][Q][K] (gradient w.r.t. the pre-epilogue conv
 * output, i.e. after the caller applied act'/mask).  For up == 2 or reflect padding the SIMT
 * path needs `workspace` of b200gan_conv2d_dgrad_workspace_floats() floats.
 * Replaces cudnnConvolutionBackwardData behind autograd of nn.Conv2d (dcgan.py:168,182). */
size_t b200gan_conv2d_dgrad_workspace_floats(const b200gan_conv_geom *g, int algo);
int b200gan_conv2d_dgrad(const b200gan_conv_geom *g, const float *dy, const float *packed,
                         float *dx, float *workspace, int algo, void *stream);

/* dw (parameter layout: Conv2d [K][C][R][S], ConvTranspose2d [C][K][R][S]) and db[K] (or NULL).
 * dw/db are OVERWRITTEN.  workspace: b200gan_conv2d_wgrad_workspace_floats() floats.
 * Replaces cudnnConvolutionBackwardFilter (dcgan.py:168,182). */
size_t b200gan_conv2d_wgrad_workspace_floats(const b200gan_conv_geom *g, int algo);
int b200gan_conv2d_wgrad(const b200gan_conv_geom *g, const float *x, const float *dy, float *dw,
                         float *db, float *workspace, int algo, void *stream);

/* dz = dy * act'(y) * chan_scale  -- backward of the fused fprop epilogue, from the saved
 * output y (LeakyReLU/ReLU sign and Tanh/Sigmoid derivative are functions of y).
 * n = N*P*Q*K elements, K channels, PQ pixels per sample (for chan_scale indexing). */
int b200gan_epilogue_bwd(const float *dy, const float *y, const float *chan_scale, int32_t act,
                         float slope, int64_t n, int32_t K, int64_t PQ, int32_t round_tf32,
                         float *dz, void *stream);

/* db[k] = sum over (n,p,q) of dy * act'(y) * chan_scale -- the bias gradient of a fused conv block computed from
 * UNROUNDED values (when dz is TF32-rounded for the tensor-core dgrad/wgrad, summing the rounded values loses the
 * cancellation a bias gradient lives on).  db is overwritten. */
int b200gan_bias_grad(const float *dy, const float *y, const float *chan_scale, int32_t act, float slope,
                      int64_t rows, int32_t K, int64_t PQ, float *db, void *stream);

/* ---- BatchNorm2d (training) / InstanceNorm2d ------------------------------------------ */
/* Normalisation over groups: G = C (per_sample == 0: BatchNorm2d, dcgan.py:53,56,60,80) or
 * N*C (per_sample == 1: InstanceNorm2d, pix2pix/models.py:25,40,117, cyclegan/models.py:29...). */
typedef struct b200gan_norm_desc {
  int32_t N, HW, C;
  int32_t per_sample;
  float eps;      /* dcgan.py:56 passes 0.8 here (second positional arg of BatchNorm2d)         */
  float momentum; /* running-stat momentum (BatchNorm2d only)                                  */
  int32_t act;    /* activation fused after the affine transform                               */
  float slope;
  int32_t round_tf32;
} b200gan_norm_desc;

/* stats[2][G] (fp64, zeroed by the caller) += (sum x, sum x^2).  Skip when the producing conv
 * already accumulated them in its epilogue. */
int b200gan_norm_stats(const b200gan_norm_desc *d, const float *x, double *stats, void *stream);
/* From stats: mean_rstd[2][G]; scale_shift[2][G] (= gamma*rstd, beta-mean*gamma*rstd; gamma,
 * beta may be NULL = 1,0); running_mean/var (may be NULL) updated with the UNBIASED variance,
 * num_batches_tracked (int64, may be NULL) += 1 -- torch.nn.BatchNorm2d semantics.
 * `stats` is CONSUMED: it is zeroed on return, so a persistent accumulator never needs a memset. */
int b200gan_norm_finalize(const b200gan_norm_desc *d, double *stats, const float *gamma,
                          const float *beta, float *mean_rstd, float *scale_shift,
                          float *running_mean, float *running_var, int64_t *num_batches_tracked,
                          void *stream);
/* y = act(x * scale + shift); may run in place (y == x). */
int b200gan_norm_apply(const b200gan_norm_desc *d, const float *x, const float *scale_shift,
                       float *y, void *stream);
/* Backward.  Inputs: dy, saved input x, mean_rstd, gamma (or NULL), and for a fused activation EITHER scale_shift
 * (LeakyReLU / ReLU: the mask is recomputed from x, nothing else has to be kept) OR the saved output y.
 * sums[2][G] fp64 workspace: zero on entry, handed back zeroed.
 * Outputs: dx; dgamma_dbeta[2][G] (only meaningful for per_sample == 0 with affine; may be NULL). */
int b200gan_norm_bwd(const b200gan_norm_desc *d, const float *dy, const float *x, const float *y,
                     const float *mean_rstd, const float *scale_shift, const float *gamma, double *sums, float *dx,
                     float *dgamma_dbeta, void *stream);
/* Double backward of training-mode BatchNorm2d (per_sample == 0 only; InstanceNorm returns an error) with an optional
 * fused LeakyReLU / ReLU: the derivative of b200gan_norm_bwd's outputs (dx, dgamma, dbeta) w.r.t. its inputs, for the
 * gradient penalty of a BatchNorm critic (autograd.grad(..., create_graph=True)).
 * Inputs: dy and x as given to b200gan_norm_bwd, u = dL/d(dx), mean_rstd, scale_shift (required for a fused activation:
 * the mask is recomputed from the sign of x * scale + shift; may be NULL without one), gamma (NULL = 1),
 * gg_gamma = dL/d(dgamma) and gg_beta = dL/d(dbeta) [C] (each may be NULL = 0).
 * sums[5][C] fp64 workspace: zero on entry, handed back zeroed.
 * Outputs, all overwritten: gx = dL/dx and gdy = dL/d(dy) [N][HW][C]; dgamma [C] = dL/dgamma (may be NULL).
 * round_tf32 is ignored: both outputs are gradients that autograd sums with other terms, not conv operands. */
int b200gan_norm_bwd_bwd(const b200gan_norm_desc *d, const float *dy, const float *x, const float *u,
                         const float *mean_rstd, const float *scale_shift, const float *gamma, const float *gg_gamma,
                         const float *gg_beta, double *sums, float *gx, float *gdy, float *dgamma, void *stream);

/* ---- Generator tail: BatchNorm2d -> LeakyReLU/ReLU -> Conv2d(C, K<=3, 3, 1, 1) -> Tanh, fused -------------- */
/* Replaces the module run dcgan.py:60-63
 *     nn.BatchNorm2d(64, 0.8), nn.LeakyReLU(0.2, inplace=True), nn.Conv2d(64, opt.channels, 3, stride=1, padding=1), nn.Tanh()
 * acting on `a`, the raw output of the preceding convolution: the normalised/activated tensor, its gradient and the
 * conv's data gradient are never written to memory (csrc/tail.cu).  scale_shift / mean_rstd come from
 * b200gan_norm_finalize (batch statistics of `a`).  Supported: C in {32, 64, 128}, K in 1..3, W a power of two in
 * [16, 128], act_mid in {NONE, LRELU, RELU}. */
typedef struct b200gan_tail_desc {
  int32_t N, H, W, C; /* a: [N][H][W][C] */
  int32_t K;          /* conv output channels; the conv is 3x3, stride 1, zero padding 1 */
  int32_t act_mid;    /* activation between the norm and the conv */
  float slope;
  int32_t act_out;    /* activation after the conv (+bias) */
} b200gan_tail_desc;
int b200gan_tail_supported(const b200gan_tail_desc *d);
/* out[N][H][W][K] = act_out(conv3x3(act_mid(a * scale + shift), w) + bias); w: the Conv2d parameter [K][C][3][3].
 * The convolution runs on tcgen05 (kind::tf32). */
int b200gan_tail_fprop(const b200gan_tail_desc *d, const float *a, const float *scale_shift, const float *w,
                       const float *bias, float *out, void *stream);
/* Backward of the same composite given g = d(loss)/d(conv output before act_out) [N][H][W][K]:
 *   da[N][H][W][C]  gradient w.r.t. `a` through conv, activation and the training-mode BatchNorm
 *   dgamma_dbeta[2][C] (may be NULL), dw[K][C][3][3], db[K] (may be NULL) -- all OVERWRITTEN.
 * workspace: b200gan_tail_bwd_workspace_bytes() bytes, 16-byte aligned (zeroed by the call). */
size_t b200gan_tail_bwd_workspace_bytes(const b200gan_tail_desc *d);
int b200gan_tail_bwd(const b200gan_tail_desc *d, const float *a, const float *mean_rstd, const float *scale_shift,
                     const float *w, const float *g, void *workspace, float *da, float *dgamma_dbeta, float *dw,
                     float *db, int32_t round_tf32, void *stream);

/* ---- shape / index ops (bit-exact) ---------------------------------------------------- */
/* NCHW <-> NHWC transposes of a dense fp32 tensor. */
int b200gan_nchw_to_nhwc(const float *x, float *y, int32_t N, int32_t C, int32_t HW, void *stream);
int b200gan_nhwc_to_nchw(const float *x, float *y, int32_t N, int32_t C, int32_t HW, void *stream);
/* Stand-alone versions of the modules that are normally folded into a conv:
 * nearest x2 upsample and its gradient (sum over the 2x2 replicas), NHWC. */
int b200gan_upsample2x_fwd(const float *x, float *y, int32_t N, int32_t H, int32_t W, int32_t C,
                           void *stream);
int b200gan_upsample2x_bwd(const float *dy, float *dx, int32_t N, int32_t H, int32_t W, int32_t C,
                           void *stream);
/* Constant-zero or reflection padding and its gradient (crop / fold), NHWC. */
/* round_tf32: store RN-rounded TF32 values (the padded copy feeds a tcgen05 conv) */
int b200gan_pad2d_fwd(const float *x, float *y, int32_t N, int32_t H, int32_t W, int32_t C,
                      int32_t pad_t, int32_t pad_l, int32_t pad_b, int32_t pad_r, int32_t mode,
                      int32_t round_tf32, void *stream);
int b200gan_pad2d_bwd(const float *dy, float *dx, int32_t N, int32_t H, int32_t W, int32_t C,
                      int32_t pad_t, int32_t pad_l, int32_t pad_b, int32_t pad_r, int32_t mode,
                      void *stream);
/* Element-wise activation (optionally times a per-element or per-(n,c) mask) and backward. */
int b200gan_act_fwd(const float *x, const float *mask, int32_t mask_per_channel, int32_t act,
                    float slope, int64_t n, int32_t C, int64_t HW, float *y, void *stream);

/* ---- WGAN-GP critic: whole gradient-penalty double backward in one kernel --------------- */
/* Critic D(x) = W3 lrelu(W2 lrelu(W1 x + b1) + b2) + b3  (wgan_gp.py:72-78), Din -> H1 -> H2 -> 1.
 * Computes, for interpolates xi[N][Din] (wgan_gp.py:124):
 *   gp = mean_n (||dD/dxi||_2 - 1)^2                                  (wgan_gp.py:128-137)
 * and, scaled by `lambda_gp` (wgan_gp.py:87,171), its gradient w.r.t. W1, W2, W3 -- the closed
 * form of autograd's double backward (SURVEY.md section 8a row a7); biases get zero gradient.
 * Outputs are OVERWRITTEN: gp[1], dW1[H1][Din], dW2[H2][H1], dW3[H2].
 * workspace: b200gan_gp_mlp_workspace_floats() floats. */
typedef struct b200gan_gp_mlp_desc {
  int32_t N, Din, H1, H2;
  float slope;
  float lambda_gp;
} b200gan_gp_mlp_desc;
size_t b200gan_gp_mlp_workspace_floats(const b200gan_gp_mlp_desc *d);
int b200gan_gp_mlp_fwd_bwd(const b200gan_gp_mlp_desc *d, const float *xi, const float *W1,
                           const float *b1, const float *W2, const float *b2, const float *W3,
                           float *gp, float *dW1, float *dW2, float *dW3, float *workspace,
                           void *stream);

/* The whole critic iteration of wgan_gp.py:164-173 for the MLP critic in ONE cooperative kernel:
 *   losses[0] = -mean(D(real)) + mean(D(fake)) + lambda * gp,   losses[1] = lambda * gp,
 * with the interpolates alpha * real + (1 - alpha) * fake formed inside (alpha [N], wgan_gp.py:122-124), and the
 * gradient of losses[0] w.r.t. every parameter of D (all OVERWRITTEN): first-order backward of the real / fake passes and
 * the closed-form double backward of the penalty share their GEMMs (csrc/gp_mlp.cu).  real, fake: [N][Din]. */
size_t b200gan_critic_step_workspace_floats(const b200gan_gp_mlp_desc *d);
int b200gan_critic_step_mlp(const b200gan_gp_mlp_desc *d, const float *real, const float *fake, const float *alpha,
                            const float *W1, const float *b1, const float *W2, const float *b2, const float *W3,
                            const float *b3, float *losses, float *dW1, float *db1, float *dW2, float *db2, float *dW3,
                            float *db3, float *workspace, void *stream);

/* ---- flat-buffer Adam (torch.optim.Adam semantics: dcgan.py:134-135) --------------------- */
/* p -= lr * mhat / (sqrt(vhat) + eps), bias-corrected with the step count read from the
 * device (step[0] is incremented by the kernel -> CUDA-graph capturable).  lr, betas and eps
 * are doubles like torch's Python-side hyper-parameters: torch forms 1 - beta, 1 - beta^t and
 * lr / (1 - beta1^t) in double and casts them to fp32 where they meet a tensor.
 * grad_scale multiplies g first (1/world_size after an all-reduce sum). */
int b200gan_adam_step(float *p, const float *g, float *m, float *v, int64_t n, double lr,
                      double beta1, double beta2, double eps, float grad_scale, float *step,
                      void *stream);

/* ---- Discriminator conv blocks as a fused chain (csrc/narrow_block.cu) -------------------------------------------- */
/* Replaces, for the narrow strided layers of dcgan.py:77-88
 *     [nn.Conv2d(in, out, 3, 2, 1), nn.LeakyReLU(0.2, inplace=True), nn.Dropout2d(0.25), nn.BatchNorm2d(out, 0.8)] x 4
 * every kernel between two convolutions: a layer stores a_l = dropout(lrelu(conv_l(x_l) + b_l)) and the batch sums of
 * a_l; the normalised tensor x_{l+1} = BN_l(a_l) is applied while the consumer gathers its operands and is never
 * written.  A BatchNorm seen from these kernels is the raw batch statistics plus its parameters: */
typedef struct b200gan_nb_bn {
  const double *stats; /* [groups][2][C] sum, sum of squares of the normalised tensor over a group's N*H*W; NULL = no
                          BatchNorm */
  const float *gamma;  /* [C] or NULL (= 1) */
  const float *beta;   /* [C] or NULL (= 0) */
  float eps;
  double count;        /* (N / groups)*H*W */
  int32_t groups;      /* <= 1: the whole batch is one BatchNorm batch.  G > 1: the batch is G equal runs of images with
                          independent batch statistics and weight gradients summed over all of them -- G forward passes of
                          the reference (dcgan.py:178-179: discriminator(real_imgs), discriminator(gen_imgs.detach())) in
                          one launch per layer; running statistics are updated G times in batch order.  Every stats / sums
                          buffer of the chain entry points then has a leading [groups] dimension. */
  int32_t reserved;
} b200gan_nb_bn;
/* 1 if the geometry can run in the fused chain (Conv2d, zero padding, stride 1/2, 3x3 or 4x4, C <= 128 (1 or a
 * multiple of 4), K a power of two in [4, 128]) */
int b200gan_nb_supported(const b200gan_conv_geom *g);
/* ... and with the batch split into `groups` statistics groups (see b200gan_nb_bn) */
int b200gan_nb_groups_supported(const b200gan_conv_geom *g, int32_t groups);
/* y = chan_scale[n,k] * act(conv(BN_in(x)) + bias): x = a_{l-1} [N][H][W][C]; packed = B200GAN_PACK_SIMT_FPROP.
 * in_bn (may be NULL): the BatchNorm between the producer and this conv, finalised in the prologue; running_mean/var and
 * num_batches_tracked (may be NULL) are updated once per call (per group, in order) with torch semantics.  groups: see
 * b200gan_nb_bn (must equal in_bn->groups when in_bn is given).  out_stats [groups][2][K] (may be NULL):
 * OVERWRITTEN with the batch sums of y for the next BatchNorm. */
int b200gan_nb_fprop(const b200gan_conv_geom *g, const b200gan_nb_bn *in_bn, float *running_mean, float *running_var,
                     int64_t *num_batches_tracked, float momentum, const float *x, const float *packed,
                     const float *bias, int32_t act, float slope, const float *chan_scale, float *y,
                     double *out_stats, int32_t groups, void *stream);
/* dz = BN_out-backward(g) * chan_scale * act'(a) and db[K] = column sums of dz (may be NULL).  g: gradient w.r.t. the
 * (virtual) BatchNorm output, or w.r.t. a itself when out_bn is NULL; sums [2][K]: sum g, sum g * ahat (complete). */
int b200gan_nb_dz(int32_t N, int64_t PQ, int32_t K, const float *g, const float *a, const float *chan_scale,
                  int32_t act, float slope, const b200gan_nb_bn *out_bn, const double *sums, float *dz, float *db,
                  void *stream);
/* dw [K][C][R][S] (OVERWRITTEN) from dz [N][P][Q][K] and x = BN_in(a_{l-1}) recomputed on the fly.  workspace:
 * b200gan_nb_wgrad_workspace_floats() floats of per-block partial slabs (summed in a fixed order: deterministic); NULL or
 * a size of 0: fp32 atomics into dw. */
size_t b200gan_nb_wgrad_workspace_floats(const b200gan_conv_geom *g);
int b200gan_nb_wgrad(const b200gan_conv_geom *g, const b200gan_nb_bn *in_bn, const float *x, const float *dz, float *dw,
                     float *workspace, void *stream);
/* g_out [N][H][W][C] = gradient w.r.t. the conv's (virtual) input; packed = B200GAN_PACK_SIMT_DGRAD.  With in_bn, a_prev
 * (= the stored input a_{l-1}) and sums [2][C]: sums is OVERWRITTEN with sum g_out, sum g_out * ahat_prev, which is what
 * the backward of the BatchNorm in front of this conv needs (and its dbeta / dgamma). */
int b200gan_nb_dgrad(const b200gan_conv_geom *g, const float *dz, const float *packed, const b200gan_nb_bn *in_bn,
                     const float *a_prev, float *g_out, double *sums, void *stream);
/* End of a chain: out = BN(a) as a real tensor, [N][C][HW] (nchw != 0: what the script's .view expects, dcgan.py:96) or
 * [N][HW][C]; and its backward: g [N][HW][C] = dout re-laid-out, sums [2][C] OVERWRITTEN. */
int b200gan_nb_tail_fwd(int32_t N, int32_t HW, int32_t C, const b200gan_nb_bn *bn, float *running_mean,
                        float *running_var, int64_t *num_batches_tracked, float momentum, const float *a, float *out,
                        int32_t nchw, void *stream);
int b200gan_nb_tail_bwd(int32_t N, int32_t HW, int32_t C, const b200gan_nb_bn *bn, const float *a, const float *dout,
                        int32_t nchw, float *g, double *sums, void *stream);

/* ---- Discriminator head and adversarial loss (csrc/head.cu) --------------------------------------------------- */
/* y[n] = act(dot(x[n], w) + b): nn.Linear(K, 1) [+ nn.Sigmoid]  (dcgan.py:92).  x [N][K] row-major. */
int b200gan_linear1_fwd(const float *x, const float *w, const float *b, float *y, int32_t N, int32_t K, int32_t act,
                        void *stream);
/* Backward from the saved output y: dx [N][K] (may be NULL), dw [K], db [1] (may be NULL) are OVERWRITTEN. */
int b200gan_linear1_bwd(const float *x, const float *w, const float *y, const float *dy, float *dx, float *dw,
                        float *db, int32_t N, int32_t K, int32_t act, void *stream);
/* torch.nn.BCELoss(), reduction 'mean', log terms clamped at -100 (dcgan.py:103,166,178-179). */
int b200gan_bce_fwd(const float *v, const float *t, float *loss, int64_t n, void *stream);
int b200gan_bce_bwd(const float *v, const float *t, const float *gout, float *dv, int64_t n, void *stream);

/* Multi-tensor form: every parameter tensor of one optimizer in ONE launch (the table travels as a kernel argument;
 * `g` is whatever tensor autograd left in param.grad).  step: TWO floats on the device, zero-initialised by the caller:
 * step[0] = number of steps taken (advanced by the last block of the launch), step[1] = internal ticket counter. */
typedef struct b200gan_adam_tensor {
  float *p;
  const float *g;
  float *m;
  float *v;
  int64_t n;
} b200gan_adam_tensor;
int b200gan_adam_multi(const b200gan_adam_tensor *tensors, int32_t count, double lr, double beta1, double beta2,
                       double eps, float grad_scale, float *step, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200GAN_H */
