/* cgan_b200.h — C-ABI of the B200 (sm_100a) GAN-step / FID engine.
 *
 * The reference (google/compare_gan) has no FFI: its seam is the Python ops library
 * (compare_gan/architectures/arch_ops.py, resnet_ops.py, gans/loss_lib.py, gans/penalty_lib.py,
 * tf.train.AdamOptimizer, tfgan FID).  Each entry point below replaces the TF library kernel(s)
 * behind one of those call sites; the citation after each declaration is the reference
 * file:line it stands in for (paths relative to /root/reference/compare_gan/).
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*.
 *  - activations float32 NHWC; conv kernels HWIO [kh,kw,cin,cout]; linear kernels [in,out]
 *    (arch_ops.py:543-546, 563-565, 583-585).
 *  - every call is asynchronous on the context's stream (cgan_ctx_set_stream); no call
 *    synchronises or allocates after warm-up (workspace grows on first use only).
 *  - return 0 on success, non-zero error code otherwise; message via cgan_last_error().
 *    Nothing throws across the ABI.  A context is not thread-safe.
 */
#ifndef CGAN_B200_H_
#define CGAN_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cgan_ctx cgan_ctx;

enum { CGAN_OK = 0, CGAN_ERR_ARG = 1, CGAN_ERR_CUDA = 2, CGAN_ERR_WORKSPACE = 3, CGAN_ERR_UNSUPPORTED = 4 };

/* ---- context ------------------------------------------------------------------------- */
int cgan_version(void);
int cgan_ctx_create(cgan_ctx** out, int device);
int cgan_ctx_destroy(cgan_ctx* ctx);
int cgan_ctx_set_stream(cgan_ctx* ctx, void* cuda_stream);          /* cudaStream_t */
int cgan_ctx_reserve_workspace(cgan_ctx* ctx, size_t bytes);        /* pre-size (never during capture) */
/* 0: exact fp32 SIMT contraction; 1: tcgen05 kind::tf32 tensor-core path where the shape allows. */
int cgan_ctx_set_math_mode(cgan_ctx* ctx, int mode);
const char* cgan_last_error(cgan_ctx* ctx);
/* number of kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t cgan_launch_count(cgan_ctx* ctx);
/* Tuning knobs and introspection (tests compare kernel variants bit for bit and ask which path a contraction took).
 *   CGAN_OPT_TC_MT      (set/get) max pixel tiles (conv) / work units (filter gradient) per tcgen05 CTA: 1 or 2.
 *   CGAN_OPT_TC_HALO    (set/get) 3x3 stride-1 tcgen05 convolutions fetch one (rows+2)-row activation box per kernel column
 *                       instead of one box per tap: 0 never, 1 where it measured faster (operand rounded in the kernel,
 *                       >= 256 output channels; default), 2 wherever the geometry allows.
 *   CGAN_OPT_TC_THIN    (set/get) 1 (default): in math_mode 1 the image-side convolutions (<= 4 input or <= 4 output channels,
 *                       kh*kw*channels <= 32: every discriminator's first and every generator's last convolution, Inception's
 *                       stem) run as ONE 32-wide GEMM on the tcgen05 kernels over a [pixels, 32] patch tensor (csrc/thin_tc.cu),
 *                       TF32 operands like every other tensor-core contraction; 0: the exact-fp32 streaming kernels (thin.cu).
 *   CGAN_OPT_LAST_PATH  (get) CGAN_PATH_* taken by the most recent conv2d_fwd / dgrad / wgrad / gemm_batched call. */
enum { CGAN_OPT_TC_MT = 1, CGAN_OPT_LAST_PATH = 2, CGAN_OPT_TC_HALO = 3, CGAN_OPT_TC_THIN = 6 };
enum { CGAN_PATH_SIMT_FP32 = 0, CGAN_PATH_TCGEN05_TF32 = 1, CGAN_PATH_THIN_FP32 = 2 };
int cgan_ctx_set_option(cgan_ctx* ctx, int key, int64_t value);
int cgan_ctx_get_option(cgan_ctx* ctx, int key, int64_t* host_value);

/* ---- utilities ------------------------------------------------------------------------ */
int cgan_fill(cgan_ctx*, float* dst, float value, int64_t n);
int cgan_copy(cgan_ctx*, float* dst, const float* src, int64_t n);
/* dst[r, dst_off + j] = src[r, src_off + j], j < cols  (tf.concat / tf.split on axis 1) */
int cgan_copy2d(cgan_ctx*, float* dst, int dst_ld, int dst_off, const float* src, int src_ld, int src_off,
                int64_t rows, int cols);
/* y = a*x + b*y0 + c   (y0 nullable) — x*2-1 (sndcgan.py:108), (tanh+1)/2, grad accumulation */
int cgan_axpby(cgan_ctx*, float* y, float a, const float* x, float b, const float* y0, float c, int64_t n);
/* y[i] = x[i] * (*scalar_dev) * mul  — non_local_block sigma (arch_ops.py:758), 1/sigma scaling */
int cgan_scale_by_dev(cgan_ctx*, float* y, const float* x, const float* scalar_dev, float mul, int inverse, int64_t n);
/* out[0] = sum_i a[i]*b[i]  (deterministic two-stage) — d sigma of non_local_block, SN backward */
int cgan_dot(cgan_ctx*, float* out_dev, const float* a, const float* b, int64_t n);
/* out[i] = uniform [0, 1) from the counter-based generator SplitMix64(seed, offset + i) (24 mantissa bits): the
 * tf.random.uniform draws of the gradient penalties (gans/penalty_lib.py:72-73) when the caller does not feed them.
 * Stateless: the same (seed, offset) always yields the same numbers, on any launch configuration. */
int cgan_random_uniform(cgan_ctx*, float* out, int64_t n, uint64_t seed, uint64_t offset);
/* y[n,:] = x[n,:] + alpha[n]*(xf[n,:]-x[n,:]) — WGAN-GP interpolates (gans/penalty_lib.py:74-75) */
int cgan_interpolate(cgan_ctx*, float* y, const float* x, const float* xf, const float* alpha, int n, int64_t per);
/* one-hot rows: out[n, labels[n]] = 1 (gans/modular_gan.py:359-363) */
int cgan_one_hot(cgan_ctx*, float* out, const int32_t* labels, int n, int classes);

/* ---- contractions ---------------------------------------------------------------------- */
typedef struct {
  int32_t n, h, w, cin;      /* real input tensor [n,h,w,cin] */
  int32_t cout, kh, kw, stride;
  int32_t upsample;          /* 1: input is zero-inserted 2x first (resnet_ops.py:35-56, :122-123), never materialised */
  int32_t oh, ow;            /* output spatial size */
  int32_t pad_t, pad_l;      /* TF SAME: before = total/2 */
} cgan_conv_desc;

/* y = conv(x, w) + bias   — tf.nn.conv2d(..., "SAME") + bias_add, arch_ops.py:568-572;
 * with desc.upsample: conv(unpool(x)), resnet_ops.py:122-130. */
int cgan_conv2d_fwd(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* w_hwio, const float* bias, float* y);
/* same with a fused activation (act = 0 or CGAN_ACT_RELU): conv + folded-BN bias + ReLU of the Inception graph
 * (tfgan.eval.run_inception, eval_utils.py:165-175); inference only. */
int cgan_conv2d_fwd_act(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* w_hwio, const float* bias, int act,
                        float* y);
/* same, writing output pixel p's `cout` channels at y + p*ldy (ldy >= cout): the convolution stores straight into its
 * channel slice of a wider NHWC tensor, which is tf.concat(axis=3) of the Inception "mixed" blocks without the copy
 * (tfgan.eval.run_inception, eval_utils.py:165-175).  Not available with desc.upsample. */
int cgan_conv2d_fwd_act_ld(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* w_hwio, const float* bias, int act,
                           float* y, int ldy);
/* dx = d/dx of the above (TF Conv2DBackpropInput); this is also tf.nn.conv2d_transpose, arch_ops.py:588-589. */
int cgan_conv2d_dgrad(cgan_ctx*, const cgan_conv_desc*, const float* dy, const float* w_hwio, float* dx);
/* dw = d/dw (TF Conv2DBackpropFilter); deterministic split-K. */
int cgan_conv2d_wgrad(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* dy, float* dw);
/* Fused forms of the three convolution entry points: what the reference writes as separate TF ops around a convolution
 * inside its residual blocks is done in the convolution's epilogue, so each activation tensor crosses HBM once:
 *   y = act(conv(x, w) + bias + residual)                 residual add of resnet_ops.py:181 / resnet_biggan.py:150
 *   act = ReLU when flags & CGAN_CONV_RELU                 tf.nn.relu of resnet_ops.py:161,174 (the consumer's pre-activation)
 *   y = mask > 0 ? y : mask_leak * y                       the (leaky-)ReLU gradient (arch_ops.py:595-597) applied to an input
 *                                                          gradient: mask is the activation's input (or output), same shape as y
 *   CGAN_CONV_ROUND_OUT: y is stored rounded to the nearest TF32 value (its only consumers are tensor-core contractions,
 *   which would round it anyway); CGAN_CONV_IN_TF32 / CGAN_CONV_IN2_TF32 assert that the first / second activation operand
 *   (x or dy; for wgrad x and dy) already holds TF32-representable values, so the kernel skips its operand-rounding pass.
 * In math_mode 0 (exact fp32) the rounding flags must not be set by the caller.  ldy: output pixel stride (0 = cout). */
enum { CGAN_CONV_RELU = 1, CGAN_CONV_ROUND_OUT = 2, CGAN_CONV_IN_TF32 = 4, CGAN_CONV_IN2_TF32 = 8 };
typedef struct {
  const float* bias;        /* [cout] (fwd) / [cin] (dgrad), nullable */
  const float* residual;    /* same shape as the output, nullable */
  const float* mask;        /* same shape as the output, nullable */
  float mask_leak;          /* 0 for ReLU, the leak for leaky ReLU */
  int32_t flags;
  int32_t ldy;
} cgan_conv_epilogue;
int cgan_conv2d_fwd_ex(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* w_hwio, const cgan_conv_epilogue* ep,
                       float* y);
int cgan_conv2d_dgrad_ex(cgan_ctx*, const cgan_conv_desc*, const float* dy, const float* w_hwio, const cgan_conv_epilogue* ep,
                         float* dx);
int cgan_conv2d_wgrad_ex(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* dy, int flags, float* dw);
/* C = alpha*op(A)*op(B) + beta*C, row-major, op = transpose when flag set — tf.matmul in
 * linear (arch_ops.py:548), projection head (resnet_biggan.py:419-423), attention (arch_ops.py:744,753). */
int cgan_gemm(cgan_ctx*, int trans_a, int trans_b, int m, int n, int k, float alpha, const float* a, int lda,
              const float* b, int ldb, float beta, float* c, int ldc);
int cgan_gemm_batched(cgan_ctx*, int trans_a, int trans_b, int m, int n, int k, float alpha, const float* a, int lda,
                      int64_t stride_a, const float* b, int ldb, int64_t stride_b, float beta, float* c, int ldc,
                      int64_t stride_c, int batch);

/* ---- fused self-attention (non_local_block, arch_ops.py:734-753) --------------------------------------------------
 * out[i] = softmax(q[i] k[i]^T) v[i] per image i: q = theta [batch, lq, dk], k = phi [batch, lk, dk], v = g [batch, lk, dv],
 * out [batch, lq, dv] — tf.matmul(theta, phi, transpose_b=True) -> tf.nn.softmax -> tf.matmul(attn, g) in ONE tcgen05
 * kernel: the [lq, lk] scores live in TMEM / shared memory only (csrc/attn_tc.cu).  lse [batch, lq] receives the
 * log-sum-exp of every score row; the backward recomputes the probabilities from it.  Operands are consumed as TF32:
 * pass tensors that already hold TF32-representable values (cgan_round_tf32, or a producer's ROUND_OUT epilogue).
 * cgan_attention_supported returns 1 when the fused kernels accept the shape in the current math mode (math_mode 1,
 * lq and lk multiples of 128, dk <= 32 and a multiple of 4, dv <= 128 and a multiple of 16), else 0 — callers then
 * compose cgan_gemm_batched / cgan_softmax_* as the reference does. */
int cgan_attention_supported(cgan_ctx*, int batch, int lq, int lk, int dk, int dv);
int cgan_attention_fwd(cgan_ctx*, const float* q, const float* k, const float* v, float* out, float* lse, int batch, int lq,
                       int lk, int dk, int dv);
/* gradients of the above w.r.t. q, k, v given dout [batch, lq, dv] (TF's MatMul / Softmax gradients of arch_ops.py:744-753):
 * two kernels, one accumulating dq per query tile, one accumulating dk and dv per key tile; fixed summation order. */
int cgan_attention_bwd(cgan_ctx*, const float* q, const float* k, const float* v, const float* out, const float* lse,
                       const float* dout, float* dq, float* dk_out, float* dv_out, int batch, int lq, int lk, int dk, int dv);
/* y = x rounded to the nearest TF32 value (10 mantissa bits), what a tensor-core contraction in math_mode 1 does to its operands */
int cgan_round_tf32(cgan_ctx*, float* y, const float* x, int64_t n);

/* ---- rows x channels reductions / bias -------------------------------------------------- */
/* y[r,c] = x[r,c] + bias[c]   (linear bias, arch_ops.py:549-555) */
int cgan_bias_add(cgan_ctx*, float* y, const float* x, const float* bias, int64_t rows, int c);
/* out[g,c] = sum over the rows of group g of x[r,c]; rows = groups*rows_per_group (bias / beta gradients) */
int cgan_colsum(cgan_ctx*, float* out, const float* x, int groups, int64_t rows_per_group, int c);

/* ---- batch norm (arch_ops.py:194-319, 327-367, 423-445; tpu/tpu_ops.py:94-125) ------------ */
/* local moments: mean[c] = sum x / rows, meansq[c] = sum x^2 / rows  (fp32; stats[0:c]=mean, stats[c:2c]=meansq).
 * Cross-replica BN all-reduces this [2c] buffer and divides by the replica count (tpu_ops.py:110-125). */
int cgan_bn_moments(cgan_ctx*, float* stats2c, const float* x, int64_t rows, int c);
/* var = meansq - mean^2 (arch_ops.py:289-297 / tpu_ops.py:125); optional moving-average update
 * m <- m - (m - batch)*(1-decay) (arch_ops.py:100-117); moving_* nullable. */
int cgan_bn_finalize(cgan_ctx*, float* mean_var2c, const float* stats2c, int c, float* moving_mean, float* moving_var,
                     float decay);
/* accumulator inference path (arch_ops.py:122-191): if *update_accus_dev==1 accumulate; write accu/counter to mean_var2c */
int cgan_bn_accumulate(cgan_ctx*, float* mean_var2c, const float* batch_mean_var2c, int c, float* accu_mean,
                       float* accu_var, float* accu_counter, const float* update_accus_dev);
/* y = (x-mean)*rsqrt(var+eps)*gamma + beta; gamma/beta: [c] (cond=0) or [samples,c] (cond=1, one row per sample of
 * rows_per_sample rows); either nullable; act: 0 none, 1 relu. */
int cgan_bn_apply(cgan_ctx*, float* y, const float* x, int64_t rows, int c, int64_t rows_per_sample,
                  const float* mean_var2c, float eps, const float* gamma, const float* beta, int cond, int act);
/* backward of training-mode BN.  Step 1 (reduce): sums2c[0:c] = sum dxhat, sums2c[c:2c] = sum dxhat*xhat over LOCAL rows
 * (all-reduced by the caller under cross-replica BN); dgamma/dbeta: [c] or [samples,c] (nullable). */
int cgan_bn_bwd_reduce(cgan_ctx*, float* sums2c, float* dgamma, float* dbeta, const float* dy, const float* x,
                       int64_t rows, int c, int64_t rows_per_sample, const float* mean_var2c, float eps,
                       const float* gamma, int cond);
/* Step 2: dx = inv*(dxhat - sums[0]/count - xhat*sums[1]/count), count = GLOBAL rows; round_tf32: store dx rounded to the
 * nearest TF32 value (it is the dy operand of the producing convolution's tensor-core gradients). */
int cgan_bn_bwd_apply(cgan_ctx*, float* dx, const float* dy, const float* x, int64_t rows, int c, int64_t rows_per_sample,
                      const float* mean_var2c, float eps, const float* gamma, int cond, const float* sums2c,
                      float inv_count, int round_tf32);

/* ---- spectral norm (arch_ops.py:453-535) -------------------------------------------------- */
/* One power iteration on w[rows,cols]; left=1: u[rows], v[cols] (arch_ops.py:505-509,525); left=0: u[cols], v[rows]
 * (:511-513,527).  u is updated in place (:516); v and sigma are outputs; wbar = w / sigma (nullable). */
int cgan_spectral_norm(cgan_ctx*, const float* w, int rows, int cols, int left, float eps, float* u_inout, float* v_out,
                       float* sigma_out, float* wbar_out);
/* The same for `n` weights in ONE launch (one CTA per weight; meant for the small kernels of a discriminator — resnet_cifar,
 * SNDCGAN — where the per-weight entry point costs ~7 launches each).  `items_dev` is a device array; item i reads w / u,
 * updates u in place and writes wbar at wbar_base + wbar_off, v at v_base + v_off, sigma at sigma_base[i] and a copy of
 * the updated u (which the backward needs; later call sites overwrite u) at u_used_base + u_off.
 * max_rows_plus_cols = max over items of rows + cols (shared-memory sizing). */
typedef struct {
  const float* w;
  float* u;
  int32_t rows, cols, left, reserved;
  int64_t wbar_off, v_off, u_off;
} cgan_sn_item;
int cgan_spectral_norm_batched(cgan_ctx*, const cgan_sn_item* items_dev, int n, int max_rows_plus_cols, float eps,
                               float* wbar_base, float* v_base, float* sigma_base, float* u_used_base);
/* dw = (dwbar - <dwbar, wbar> * outer) / sigma, outer = u v^T (left) or v u^T (right); u,v constants (:521-522). */
int cgan_spectral_norm_bwd(cgan_ctx*, float* dw, const float* dwbar, const float* wbar, int rows, int cols, int left,
                           const float* u, const float* v, const float* sigma);

/* ---- pointwise / pooling ------------------------------------------------------------------- */
enum { CGAN_ACT_RELU = 1, CGAN_ACT_LRELU = 2, CGAN_ACT_SIGMOID = 3, CGAN_ACT_TANH01 = 4 /* (tanh(x)+1)/2 */ };
/* OR-ed into `kind` (act_fwd / act_bwd) or `act` (bn_apply): store the result rounded to the nearest TF32 value — the
 * tensor only feeds tensor-core contractions, which then skip their own operand-rounding pass (math_mode 1 only). */
enum { CGAN_ACT_ROUND_TF32 = 0x100 };
int cgan_act_fwd(cgan_ctx*, float* y, const float* x, int kind, float leak, int64_t n);
/* dx = dy * act'(.) ; `ref` is x for relu/lrelu and y for sigmoid/tanh01 */
int cgan_act_bwd(cgan_ctx*, float* dx, const float* dy, const float* ref, int kind, float leak, int64_t n);
int cgan_add(cgan_ctx*, float* y, const float* a, const float* b, int64_t n);
/* same, optionally storing TF32-rounded sums (gradient accumulation in front of a tensor-core contraction) */
int cgan_add_tf32(cgan_ctx*, float* y, const float* a, const float* b, int64_t n, int round_tf32);
/* 2x2 stride-2 average pool (resnet_ops.py:131-133) and its adjoint */
int cgan_avgpool2_fwd(cgan_ctx*, float* y, const float* x, int n, int h, int w, int c);
int cgan_avgpool2_bwd(cgan_ctx*, float* dx, const float* dy, int n, int h, int w, int c);
/* 2x2 stride-2 max pool (arch_ops.py:741,750) and backward (first-max wins, as TF MaxPoolGrad) */
int cgan_maxpool2_fwd(cgan_ctx*, float* y, const float* x, int n, int h, int w, int c);
int cgan_maxpool2_bwd(cgan_ctx*, float* dx, const float* dy, const float* x, int n, int h, int w, int c);
/* generic k x k pooling, TF semantics: mode 0 = max, 1 = average that EXCLUDES padded cells from the divisor (tf.nn.avg_pool
 * "SAME"); pad_t/pad_l = leading padding (0 for "VALID"); oh/ow given by the caller.  Inception-v3 feature extractor
 * (tfgan.eval.run_inception, eval_utils.py:165-175). */
int cgan_pool2d_fwd(cgan_ctx*, float* y, const float* x, int n, int h, int w, int c, int k, int stride, int pad_t, int pad_l,
                    int oh, int ow, int mode);
/* global pool over h*w: out[n,c] = scale * sum_hw x (mean: resnet_cifar.py:156; sum: resnet_biggan.py:405) */
int cgan_globalpool_fwd(cgan_ctx*, float* y, const float* x, int n, int hw, int c, float scale);
int cgan_globalpool_bwd(cgan_ctx*, float* dx, const float* dy, int n, int hw, int c, float scale);
/* row softmax (tf.nn.softmax, arch_ops.py:745) and its backward */
int cgan_softmax_fwd(cgan_ctx*, float* y, const float* x, int64_t rows, int cols);
int cgan_softmax_bwd(cgan_ctx*, float* dx, const float* dy, const float* y, int64_t rows, int cols);
/* out[r] = sum_j a[r,j]*b[r,j]  (projection discriminator, resnet_biggan.py:423) */
int cgan_rowdot(cgan_ctx*, float* out, const float* a, const float* b, int64_t rows, int cols);
/* y[r,j] = a[r,j] * s[r] */
int cgan_rowscale(cgan_ctx*, float* y, const float* a, const float* s, int64_t rows, int cols);

/* ---- losses and penalties ------------------------------------------------------------------ */
enum { CGAN_LOSS_NON_SATURATING = 0, CGAN_LOSS_HINGE = 1, CGAN_LOSS_WASSERSTEIN = 2, CGAN_LOSS_LEAST_SQUARES = 3 };
/* gans/loss_lib.py:53-148.  out4 = {d_loss, d_loss_real, d_loss_fake, g_loss}.  dlogits[2b] (nullable) receives
 * d(d_loss)/dlogit (which=0) or d(g_loss)/dlogit (which=1) for the [real; fake] logit vector. */
int cgan_gan_loss(cgan_ctx*, int kind, const float* logits_real, const float* logits_fake, int b, float* out4,
                  float* dlogits, int which);
/* gans/penalty_lib.py:78-81: slopes = sqrt(1e-4 + sum_hwc g^2); penalty = mean((slopes-1)^2);
 * dg (nullable) = d(weight*penalty)/dg. */
int cgan_gp_penalty(cgan_ctx*, float* penalty_out, float* dg, const float* g, int n, int64_t per, float weight);

/* ---- self-supervision (gans/ssgan.py, gans/utils.py:38-49) ------------------------------------------------------ */
/* y = x rotated by k * 90 degrees (k = 1, 2, 3), square NHWC images: rotate_images' transposes / flips in one pass. */
int cgan_rot90(cgan_ctx*, float* y, const float* x, int n, int hw, int c, int k);
/* rotation loss: `rows` = num_rotations * m logit rows [rows, num_rotations], row r labelled r / m;
 * *loss_out = -mean log(softmax(logits)[label] + 1e-10) (ssgan.py:205-213); dlogits (nullable) = its gradient. */
int cgan_rotation_loss(cgan_ctx*, float* loss_out, float* dlogits, const float* logits, int rows, int num_rotations);

/* ---- S3GAN heads (gans/s3gan.py) --------------------------------------------------------------------------------------
 * out[r] = 1 if sum_j y[r, j] > 0.5 else 0: "is a label available for this example" (s3gan.py:121-122). */
int cgan_row_has_label(cgan_ctx*, float* out, const float* y, int rows, int cols);
/* out[r, :] = one_hot(argmax_j logits[r, j]) (first maximum wins, like tf.argmax): the predictor's hard labels
 * (s3gan.py:149-150). */
int cgan_argmax_one_hot(cgan_ctx*, float* out, const float* logits, int rows, int cols);
/* tf.losses.softmax_cross_entropy(onehot_labels = labels, logits, weights) with its default SUM_BY_NONZERO_WEIGHTS reduction
 * (s3gan.py:312-313): *loss_out = sum_r w_r * (-sum_j labels[r,j] log softmax(logits_r)_j) / max(#{w_r != 0}, 1); labels may
 * be soft; weights [rows] nullable (= 1).  dlogits (nullable) receives d loss / d logits. */
int cgan_softmax_xent(cgan_ctx*, float* loss_out, float* dlogits, const float* logits, const float* labels,
                      const float* weights, int rows, int cols);

/* ---- optimizer (tf.train.AdamOptimizer + tf.train.ExponentialMovingAverage, gans/modular_gan.py:498-508) ---- */
/* One fused multi-tensor step over a flat parameter buffer.  *step_dev (int32, device) is incremented first; then
 * lr_t = lr*sqrt(1-b2^t)/(1-b1^t); m,v updated; p -= lr_t*m/(sqrt(v)+eps).  If ema != NULL:
 * ema <- ema - (ema-p)*(1-d), d = ema_decay*[ (t-1) >= ema_start_step ]. grad_scale multiplies g first (1/world). */
int cgan_adam_step(cgan_ctx*, float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                   float eps, float grad_scale, int32_t* step_dev, float* ema, float ema_decay, int32_t ema_start_step);

/* ---- FID statistics (tfgan frechet_classifier_distance_from_activations, metrics/fid_score.py:49-51) ---- */
/* sum[d] += sum_n act[n,d]; sumxxT[d,d] += act^T act, accumulated in float64 on device. */
int cgan_cov_accumulate(cgan_ctx*, const float* act, int n, int d, double* sum, double* sumxxT);
/* bilinear resize NHWC [n,h,w,c] -> [n,oh,ow,c] (tf.image.resize_bilinear, align_corners=False) then (x*255-128)/128
 * when `inception_scale` (eval_utils.py:157-175). */
int cgan_resize_bilinear(cgan_ctx*, float* y, const float* x, int n, int h, int w, int c, int oh, int ow, int inception_scale);

/* ---- cross-replica exchange of small vectors (tpu/tpu_ops.py:75-125: cross_replica_mean / cross_replica_moments) ---- */
/* One process per GPU on one node.  Every rank allocates a communication buffer and publishes its cudaIpc handle
 * (cgan_p2p_local_handle -> 64 bytes), the host code all-gathers the handles (torch.distributed) and hands all of them
 * to cgan_p2p_connect, which maps the peers' buffers.  cgan_allreduce_small then sums x[0..n) over the ranks IN PLACE
 * with one kernel launch over NVLink peer memory (n <= cgan_p2p_max_floats()): every rank stores its vector into every
 * peer's buffer, flags it, waits for the others' flags and adds the vectors in rank order — bit-identical results on all
 * ranks, capturable into a CUDA graph.  Gradients (MBs) stay on NCCL (gans/modular_gan.py:606-616). */
int cgan_p2p_max_floats(void);
int cgan_p2p_local_handle(cgan_ctx*, int world, void* host_handle64);
int cgan_p2p_connect(cgan_ctx*, int rank, int world, const void* host_handles);
int cgan_allreduce_small(cgan_ctx*, float* x, int n);

/* ---- input pipeline (ImageDatasetV2.train_input_fn, datasets.py:261-291; host side, no GPU work) ---- */
/* The tf.data chain of the reference: repeat() -> shuffle(buffer, seed) -> batch(drop_remainder=True) -> prefetch, with
 * _parse_fn's uint8 -> float32 / 255 (datasets.py:225-227), run by a producer thread into a ring of `ring` batch buffers
 * (page-locked when a CUDA device is present, so the caller's cudaMemcpyAsync overlaps the previous step).
 * Source: `n` images NHWC contiguous in host memory, uint8 (src_dtype 0, scaled by 1/255) or float32 (src_dtype 1, copied;
 * the reference's fake data set, datasets.py:136-145), and optional int32 labels; caller-owned, must outlive the loader
 * (e.g. an mmap of a shard file).  shuffle_buffer <= 1 disables shuffling.  The shuffle is tf.data's algorithm (a buffer
 * of `shuffle_buffer` elements, each output drawn uniformly from it and replaced by the next input) on a SplitMix64
 * stream; the element ORDER is therefore not TF's (its Philox stream is not restated). */
typedef struct cgan_loader cgan_loader;
int cgan_loader_create(cgan_loader** out, const void* images, int src_dtype, const int32_t* labels, int64_t n, int h, int w,
                       int c, int batch, int shuffle_buffer, uint64_t seed, int ring);
/* Blocks until the next batch is ready: images float32 [batch,h,w,c], labels int32 [batch] (zeros without source
 * labels).  The buffers stay untouched until released; with every ring slot outstanding the call fails instead of
 * dead-locking. */
int cgan_loader_next(cgan_loader*, const float** images, const int32_t** labels);
/* Hands the `count` oldest outstanding batches back to the producer (call once their host->device copies finished). */
int cgan_loader_release(cgan_loader*, int count);
int cgan_loader_destroy(cgan_loader*);
const char* cgan_loader_last_error(cgan_loader*);

#ifdef __cplusplus
}
#endif
#endif  /* CGAN_B200_H_ */
