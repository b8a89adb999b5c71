// Context management plus the HBM-bound pointwise / pooling / loss / optimizer kernels.
// All are grid-stride loops over NHWC float32 with the channel index fastest (coalesced), sized to
// a multiple of the SM count.
//
// Replaces: tf.nn.relu / lrelu (arch_ops.py:595-597) / sigmoid / tanh, tf.nn.pool AVG
// (resnet_ops.py:131-133), max_pooling2d (arch_ops.py:741,750), reduce_mean/sum over [1,2]
// (resnet_cifar.py:156, resnet_biggan.py:405), tf.nn.softmax (arch_ops.py:745), the losses
// (gans/loss_lib.py:53-148), the WGAN-GP slope penalty (gans/penalty_lib.py:78-81) and
// tf.train.AdamOptimizer + ExponentialMovingAverage (gans/modular_gan.py:498-508).
#include "common.cuh"

// ---------------------------------------------------------------------------------------- context
int cgan_version(void) { return 1; }

int cgan_ctx_create(cgan_ctx** out, int device) {
  if (!out) return CGAN_ERR_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return CGAN_ERR_CUDA;
  cgan_ctx* c = new cgan_ctx();
  memset(c, 0, sizeof(*c));
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess) { delete c; return CGAN_ERR_CUDA; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return CGAN_ERR_CUDA; }
  c->num_sms = prop.multiProcessorCount;
  c->tc_mt_max = 2;
  c->tc_halo = 1;
  c->tc_thin = 1;
  c->stream = 0;
  if (cudaMalloc(reinterpret_cast<void**>(&c->counters), CGAN_NUM_COUNTERS * sizeof(unsigned)) != cudaSuccess ||
      cudaMemset(c->counters, 0, CGAN_NUM_COUNTERS * sizeof(unsigned)) != cudaSuccess) {
    c->counters = nullptr;          // reductions fall back to their two-launch form
    cudaGetLastError();
  }
  *out = c;
  return CGAN_OK;
}

int cgan_ctx_destroy(cgan_ctx* ctx) {
  if (!ctx) return CGAN_ERR_ARG;
  if (ctx->ws) cudaFree(ctx->ws);
  if (ctx->counters) cudaFree(ctx->counters);
  delete ctx;
  return CGAN_OK;
}

int cgan_ctx_set_stream(cgan_ctx* ctx, void* s) {
  if (!ctx) return CGAN_ERR_ARG;
  ctx->stream = reinterpret_cast<cudaStream_t>(s);
  return CGAN_OK;
}

int cgan_ctx_reserve_workspace(cgan_ctx* ctx, size_t bytes) {
  if (!ctx) return CGAN_ERR_ARG;
  void* p;
  return cgan_ws(ctx, bytes, &p);
}

int cgan_ctx_set_math_mode(cgan_ctx* ctx, int mode) {
  if (!ctx) return CGAN_ERR_ARG;
  CGAN_REQUIRE(ctx, mode == 0 || mode == 1, "mode must be 0 (fp32 SIMT) or 1 (tcgen05 tf32)");
  ctx->math_mode = mode;
  return CGAN_OK;
}

int cgan_ctx_set_option(cgan_ctx* ctx, int key, int64_t value) {
  if (!ctx) return CGAN_ERR_ARG;
  switch (key) {
    case CGAN_OPT_TC_MT:
      CGAN_REQUIRE(ctx, value == 1 || value == 2, "CGAN_OPT_TC_MT must be 1 or 2");
      ctx->tc_mt_max = (int)value;
      return CGAN_OK;
    case CGAN_OPT_TC_HALO:
      CGAN_REQUIRE(ctx, value >= 0 && value <= 2, "CGAN_OPT_TC_HALO must be 0, 1 or 2");
      ctx->tc_halo = (int)value;
      return CGAN_OK;
    case CGAN_OPT_TC_THIN:
      CGAN_REQUIRE(ctx, value == 0 || value == 1, "CGAN_OPT_TC_THIN must be 0 or 1");
      ctx->tc_thin = (int)value;
      return CGAN_OK;
    default:
      return cgan_fail(ctx, CGAN_ERR_ARG, "%s: unknown or read-only option%s", "cgan_ctx_set_option");
  }
}

int cgan_ctx_get_option(cgan_ctx* ctx, int key, int64_t* host_value) {
  if (!ctx) return CGAN_ERR_ARG;
  CGAN_REQUIRE(ctx, host_value, "null pointer");
  switch (key) {
    case CGAN_OPT_TC_MT: *host_value = ctx->tc_mt_max; return CGAN_OK;
    case CGAN_OPT_LAST_PATH: *host_value = ctx->last_path; return CGAN_OK;
    case CGAN_OPT_TC_HALO: *host_value = ctx->tc_halo; return CGAN_OK;
    case CGAN_OPT_TC_THIN: *host_value = ctx->tc_thin; return CGAN_OK;
    default:
      return cgan_fail(ctx, CGAN_ERR_ARG, "%s: unknown option%s", "cgan_ctx_get_option");
  }
}

const char* cgan_last_error(cgan_ctx* ctx) { return ctx ? ctx->err : "null context"; }
int64_t cgan_launch_count(cgan_ctx* ctx) { return ctx ? ctx->launches : -1; }

namespace {

inline int ew_grid(cgan_ctx* ctx, long long n) {
  long long b = (n + 255) / 256;
  long long cap = (long long)ctx->num_sms * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

#define EW_LOOP(i, n)                                                                  \
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x, s__ = (long long)gridDim.x * blockDim.x; \
       i < (n); i += s__)

__global__ void fill_kernel(float* d, float v, long long n) { EW_LOOP(i, n) d[i] = v; }
__global__ void copy_kernel(float* __restrict__ d, const float* __restrict__ s, long long n) { EW_LOOP(i, n) d[i] = s[i]; }
__global__ void copy2d_kernel(float* __restrict__ d, int dld, int doff, const float* __restrict__ s, int sld, int soff,
                              long long rows, int cols) {
  long long n = rows * cols;
  EW_LOOP(i, n) {
    long long r = i / cols;
    int j = (int)(i % cols);
    d[r * dld + doff + j] = s[r * sld + soff + j];
  }
}
__global__ void axpby_kernel(float* __restrict__ y, float a, const float* __restrict__ x, float b,
                             const float* __restrict__ y0, float c, long long n) {
  EW_LOOP(i, n) {
    float v = a * x[i] + c;
    if (y0) v += b * y0[i];
    y[i] = v;
  }
}
__global__ void scale_by_dev_kernel(float* __restrict__ y, const float* __restrict__ x, const float* s, float mul, int inv,
                                    long long n) {
  float f = inv ? mul / *s : mul * *s;
  // division by sigma is done per element to match "w / norm_value" (arch_ops.py:531) bit for bit
  if (inv && mul == 1.0f) {
    float sv = *s;
    EW_LOOP(i, n) y[i] = x[i] / sv;
  } else {
    EW_LOOP(i, n) y[i] = x[i] * f;
  }
}
__global__ void dot_partial_kernel(float* part, const float* __restrict__ a, const float* __restrict__ b, long long n) {
  __shared__ float sh[32];
  float s = 0.f;
  EW_LOOP(i, n) s += a[i] * b[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void sum_final_kernel(float* out, const float* part, int n, float scale) {
  __shared__ float sh[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s += part[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) *out = s * scale;
}
__global__ void interpolate_kernel(float* __restrict__ y, const float* __restrict__ x, const float* __restrict__ xf,
                                   const float* __restrict__ alpha, long long per, long long n) {
  EW_LOOP(i, n) {
    float a = alpha[i / per];
    y[i] = x[i] + a * (xf[i] - x[i]);
  }
}
__global__ void one_hot_kernel(float* out, const int32_t* labels, int n, int classes) {
  long long tot = (long long)n * classes;
  EW_LOOP(i, tot) {
    int r = (int)(i / classes), c = (int)(i % classes);
    out[i] = (labels[r] == c) ? 1.0f : 0.0f;
  }
}
__global__ void bias_add_kernel(float* __restrict__ y, const float* __restrict__ x, const float* __restrict__ b,
                                long long n, int c) {
  EW_LOOP(i, n) y[i] = x[i] + b[i % c];
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float rna_tf32_(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
__device__ __forceinline__ float act_fwd_1(float v, int kind, float leak) {
  if (kind == CGAN_ACT_RELU) return fmaxf(v, 0.f);
  if (kind == CGAN_ACT_LRELU) return fmaxf(v, leak * v);
  if (kind == CGAN_ACT_SIGMOID) return sigmoidf_(v);
  return (tanhf(v) + 1.0f) * 0.5f;
}
__device__ __forceinline__ float act_bwd_1(float g, float r, int kind, float leak) {
  if (kind == CGAN_ACT_RELU) return r > 0.f ? g : 0.f;
  if (kind == CGAN_ACT_LRELU) return (r > leak * r) ? g : ((r < leak * r) ? leak * g : 0.5f * (1.0f + leak) * g);
  if (kind == CGAN_ACT_SIGMOID) return g * r * (1.0f - r);
  float t = 2.0f * r - 1.0f;       // y=(tanh+1)/2 -> tanh = 2y-1
  return g * 0.5f * (1.0f - t * t);
}
// float4 bodies (n4 = n / 4 vectors) plus a scalar tail for the last n % 4 elements; `rnd`: store TF32-rounded values
__global__ void act_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int kind, float leak, long long n, int rnd) {
  const long long n4 = ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x)) & 15) ? 0 : n >> 2;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  float4* y4 = reinterpret_cast<float4*>(y);
  EW_LOOP(i, n4) {
    float4 v = x4[i];
    v.x = act_fwd_1(v.x, kind, leak); v.y = act_fwd_1(v.y, kind, leak); v.z = act_fwd_1(v.z, kind, leak); v.w = act_fwd_1(v.w, kind, leak);
    if (rnd) { v.x = rna_tf32_(v.x); v.y = rna_tf32_(v.y); v.z = rna_tf32_(v.z); v.w = rna_tf32_(v.w); }
    y4[i] = v;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v = act_fwd_1(x[i], kind, leak);
    y[i] = rnd ? rna_tf32_(v) : v;
  }
}
__global__ void act_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dy, const float* __restrict__ ref,
                               int kind, float leak, long long n, int rnd) {
  const long long n4 =
      ((reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(ref)) & 15) ? 0 : n >> 2;
  const float4* g4 = reinterpret_cast<const float4*>(dy);
  const float4* r4 = reinterpret_cast<const float4*>(ref);
  float4* o4 = reinterpret_cast<float4*>(dx);
  EW_LOOP(i, n4) {
    float4 g = g4[i], r = r4[i];
    g.x = act_bwd_1(g.x, r.x, kind, leak); g.y = act_bwd_1(g.y, r.y, kind, leak);
    g.z = act_bwd_1(g.z, r.z, kind, leak); g.w = act_bwd_1(g.w, r.w, kind, leak);
    if (rnd) { g.x = rna_tf32_(g.x); g.y = rna_tf32_(g.y); g.z = rna_tf32_(g.z); g.w = rna_tf32_(g.w); }
    o4[i] = g;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float g = act_bwd_1(dy[i], ref[i], kind, leak);
    dx[i] = rnd ? rna_tf32_(g) : g;
  }
}
// generic tail of the fused convolution entry points on the exact-fp32 paths: y = round(mask(relu(y + residual)))
__global__ void conv_post_kernel(float* __restrict__ y, long long rows, int c, int ld, const float* __restrict__ residual,
                                 const float* __restrict__ mask, float leak, int relu, int round_out) {
  long long n = rows * c;
  EW_LOOP(i, n) {
    long long r = i / c;
    long long o = r * ld + (i - r * c);
    float v = y[o];
    if (residual) v += residual[o];
    if (relu) v = fmaxf(v, 0.f);
    if (mask) v = mask[o] > 0.f ? v : leak * v;
    if (round_out) v = rna_tf32_(v);
    y[o] = v;
  }
}
// y = images rotated by k * 90 degrees as gans/utils.py:38-49 composes them from transposes and flips (square images):
// k=1: y[i][j] = x[j][h-1-i];  k=2: y[i][j] = x[h-1-i][w-1-j];  k=3: y[i][j] = x[h-1-j][i]
__global__ void rot90_kernel(float* __restrict__ y, const float* __restrict__ x, int n, int hw, int c, int k) {
  const long long tot = (long long)n * hw * hw * c;
  EW_LOOP(i, tot) {
    const int ch = (int)(i % c);
    long long t = i / c;
    const int j = (int)(t % hw); t /= hw;
    const int r = (int)(t % hw);
    const long long img = t / hw;
    int sr, sc;
    if (k == 1) { sr = j; sc = hw - 1 - r; }
    else if (k == 2) { sr = hw - 1 - r; sc = hw - 1 - j; }
    else { sr = hw - 1 - j; sc = r; }
    y[i] = x[((img * hw + sr) * hw + sc) * c + ch];
  }
}
// rotation self-supervision loss (gans/ssgan.py:205-213): rows = 4 * m logits rows, row r carries label r / m;
// loss = -mean_r log(softmax(logits_r)[label_r] + 1e-10); dlogits (nullable) = d loss / d logits.  One block.
__global__ void rotation_loss_kernel(float* loss, float* dlogits, const float* __restrict__ logits, int rows, int nrot) {
  __shared__ float sh[32];
  const int m = rows / nrot;
  float acc = 0.f;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) {
    const float* z = logits + (long long)r * nrot;
    float mx = z[0];
    for (int q = 1; q < nrot; ++q) mx = fmaxf(mx, z[q]);
    float den = 0.f;
    for (int q = 0; q < nrot; ++q) den += expf(z[q] - mx);
    const int lab = r / m;
    const float py = expf(z[lab] - mx) / den;
    acc += -logf(py + 1e-10f);
    if (dlogits) {
      const float coef = -(py / (py + 1e-10f)) / rows;          // d(-log(p_y + eps)) / dz_q = -(p_y / (p_y + eps)) (delta_qy - p_q)
      for (int q = 0; q < nrot; ++q) {
        const float pq = expf(z[q] - mx) / den;
        dlogits[(long long)r * nrot + q] = coef * ((q == lab ? 1.f : 0.f) - pq);
      }
    }
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) *loss = acc / rows;
}
// S3GAN heads (gans/s3gan.py:121-122, 149-150, 312-313); rows = examples of one sub-step, cols = classes
__global__ void row_has_label_kernel(float* __restrict__ out, const float* __restrict__ y, int rows, int cols) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int j = 0; j < cols; ++j) s += y[(long long)r * cols + j];
    out[r] = s > 0.5f ? 1.f : 0.f;
  }
}
__global__ void argmax_one_hot_kernel(float* __restrict__ out, const float* __restrict__ z, int rows, int cols) {
  for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
    const float* row = z + (long long)r * cols;
    int best = 0;
    for (int j = 1; j < cols; ++j)
      if (row[j] > row[best]) best = j;
    for (int j = 0; j < cols; ++j) out[(long long)r * cols + j] = j == best ? 1.f : 0.f;
  }
}
// one block: weighted soft-label cross entropy, SUM_BY_NONZERO_WEIGHTS
__global__ void softmax_xent_kernel(float* loss, float* dlogits, const float* __restrict__ z, const float* __restrict__ lab,
                                    const float* __restrict__ w, int rows, int cols) {
  __shared__ float sh[32];
  float acc = 0.f, present = 0.f;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) present += (w ? w[r] : 1.f) != 0.f ? 1.f : 0.f;
  present = block_sum(present, sh);
  const float inv = present > 0.f ? 1.f / present : 0.f;
  for (int r = threadIdx.x; r < rows; r += blockDim.x) {
    const float* zr = z + (long long)r * cols;
    const float* lr = lab + (long long)r * cols;
    float mx = zr[0];
    for (int j = 1; j < cols; ++j) mx = fmaxf(mx, zr[j]);
    float den = 0.f, lsum = 0.f, dot = 0.f;
    for (int j = 0; j < cols; ++j) { den += expf(zr[j] - mx); lsum += lr[j]; dot += lr[j] * (zr[j] - mx); }
    const float lden = logf(den);
    const float wr = w ? w[r] : 1.f;
    acc += wr * (lsum * lden - dot);                   // -sum_j l_j (z_j - mx - log den)
    if (dlogits)
      for (int j = 0; j < cols; ++j) dlogits[(long long)r * cols + j] = wr * inv * (lsum * expf(zr[j] - mx) / den - lr[j]);
  }
  acc = block_sum(acc, sh);
  if (threadIdx.x == 0) *loss = acc * inv;
}
__global__ void add_kernel(float* __restrict__ y, const float* __restrict__ a, const float* __restrict__ b, long long n, int rnd) {
  const long long n4 =
      ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) ? 0 : n >> 2;
  const float4* a4 = reinterpret_cast<const float4*>(a);
  const float4* b4 = reinterpret_cast<const float4*>(b);
  float4* y4 = reinterpret_cast<float4*>(y);
  EW_LOOP(i, n4) {
    float4 u = a4[i], v = b4[i];
    u.x += v.x; u.y += v.y; u.z += v.z; u.w += v.w;
    if (rnd) { u.x = rna_tf32_(u.x); u.y = rna_tf32_(u.y); u.z = rna_tf32_(u.z); u.w = rna_tf32_(u.w); }
    y4[i] = u;
  }
  for (long long i = n4 * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float v = a[i] + b[i];
    y[i] = rnd ? rna_tf32_(v) : v;
  }
}
__global__ void avgpool2_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int n, int h, int w, int c) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * oh * ow * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    const float* p = x + (((b * h + 2 * oy) * w) + 2 * ox) * c + ch;
    y[i] = (p[0] + p[c] + p[(long long)w * c] + p[(long long)w * c + c]) * 0.25f;
  }
}
__global__ void avgpool2_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dy, int n, int h, int w, int c) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * h * w * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int xx = (int)(t % w); t /= w;
    int yy = (int)(t % h);
    long long b = t / h;
    dx[i] = 0.25f * dy[(((b * oh + yy / 2) * ow) + xx / 2) * c + ch];
  }
}
// 4-channel vectorised variants (C % 4 == 0): one thread per pooled pixel x channel quad.  The scalar kernels above are
// instruction-bound (five integer divisions per element); these do the index arithmetic once per 16 output floats.
__global__ void avgpool2_fwd_v4_kernel(float4* __restrict__ y, const float4* __restrict__ x, int n, int h, int w, int c4) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * oh * ow * c4;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c4);
    long long t = i / c4;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    const float4* p = x + (((b * h + 2 * oy) * w) + 2 * ox) * c4 + ch;
    float4 a = p[0], bb = p[c4], cc = p[(long long)w * c4], d = p[(long long)w * c4 + c4];
    y[i] = make_float4((a.x + bb.x + cc.x + d.x) * 0.25f, (a.y + bb.y + cc.y + d.y) * 0.25f,
                       (a.z + bb.z + cc.z + d.z) * 0.25f, (a.w + bb.w + cc.w + d.w) * 0.25f);
  }
}
__global__ void avgpool2_bwd_v4_kernel(float4* __restrict__ dx, const float4* __restrict__ dy, int n, int h, int w, int c4) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * oh * ow * c4;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c4);
    long long t = i / c4;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    float4 g = dy[i];
    g.x *= 0.25f; g.y *= 0.25f; g.z *= 0.25f; g.w *= 0.25f;
    float4* p = dx + (((b * h + 2 * oy) * w) + 2 * ox) * c4 + ch;
    p[0] = g; p[c4] = g; p[(long long)w * c4] = g; p[(long long)w * c4 + c4] = g;
  }
}

__global__ void maxpool2_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int n, int h, int w, int c) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * oh * ow * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    const float* p = x + (((b * h + 2 * oy) * w) + 2 * ox) * c + ch;
    y[i] = fmaxf(fmaxf(p[0], p[c]), fmaxf(p[(long long)w * c], p[(long long)w * c + c]));
  }
}
__global__ void maxpool2_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dy, const float* __restrict__ x,
                                    int n, int h, int w, int c) {
  int oh = h / 2, ow = w / 2;
  long long tot = (long long)n * oh * ow * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    long long base = (((b * h + 2 * oy) * w) + 2 * ox) * c + ch;
    long long offs[4] = {0, c, (long long)w * c, (long long)w * c + c};
    int best = 0;
    float bv = x[base];
#pragma unroll
    for (int k = 1; k < 4; ++k) {
      float v = x[base + offs[k]];
      if (v > bv) { bv = v; best = k; }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) dx[base + offs[k]] = (k == best) ? dy[i] : 0.f;
  }
}
__global__ void pool2d_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int n, int h, int w, int c, int k,
                                  int stride, int pad_t, int pad_l, int oh, int ow, int mode) {
  long long tot = (long long)n * oh * ow * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    float acc = mode == 0 ? -INFINITY : 0.f;
    int cnt = 0;
    for (int dy = 0; dy < k; ++dy) {
      int iy = oy * stride + dy - pad_t;
      if (iy < 0 || iy >= h) continue;
      for (int dx = 0; dx < k; ++dx) {
        int ix = ox * stride + dx - pad_l;
        if (ix < 0 || ix >= w) continue;
        float v = x[((b * h + iy) * w + ix) * c + ch];
        acc = mode == 0 ? fmaxf(acc, v) : acc + v;
        ++cnt;
      }
    }
    y[i] = mode == 0 ? acc : acc / (float)max(cnt, 1);
  }
}
__global__ void pool2d_fwd_v4_kernel(float4* __restrict__ y, const float4* __restrict__ x, int n, int h, int w, int c4, int k,
                                     int stride, int pad_t, int pad_l, int oh, int ow, int mode) {
  long long tot = (long long)n * oh * ow * c4;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c4);
    long long t = i / c4;
    int ox = (int)(t % ow); t /= ow;
    int oy = (int)(t % oh);
    long long b = t / oh;
    float4 acc = mode == 0 ? make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY) : make_float4(0.f, 0.f, 0.f, 0.f);
    int cnt = 0;
    for (int dy = 0; dy < k; ++dy) {
      int iy = oy * stride + dy - pad_t;
      if (iy < 0 || iy >= h) continue;
      for (int dx = 0; dx < k; ++dx) {
        int ix = ox * stride + dx - pad_l;
        if (ix < 0 || ix >= w) continue;
        float4 v = x[((b * h + iy) * w + ix) * c4 + ch];
        if (mode == 0) { acc.x = fmaxf(acc.x, v.x); acc.y = fmaxf(acc.y, v.y); acc.z = fmaxf(acc.z, v.z); acc.w = fmaxf(acc.w, v.w); }
        else { acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w; }
        ++cnt;
      }
    }
    if (mode != 0) { float inv = 1.0f / (float)max(cnt, 1); acc.x *= inv; acc.y *= inv; acc.z *= inv; acc.w *= inv; }
    y[i] = acc;
  }
}
// y[n,c] = scale * sum_hw x[n,hw,c]: one thread per (n,c) strides over hw; consecutive threads -> consecutive c
__global__ void globalpool_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int n, int hw, int c, float scale) {
  long long tot = (long long)n * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long b = i / c;
    const float* p = x + b * hw * c + ch;
    float s = 0.f;
    for (int k = 0; k < hw; ++k) s += p[(long long)k * c];
    y[i] = s * scale;
  }
}
__global__ void globalpool_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dy, int n, int hw, int c, float scale) {
  long long tot = (long long)n * hw * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long b = i / ((long long)hw * c);
    dx[i] = scale * dy[b * c + ch];
  }
}
// one block per row
__global__ void softmax_fwd_kernel(float* __restrict__ y, const float* __restrict__ x, int cols) {
  __shared__ float sh[32];
  const float* xr = x + (long long)blockIdx.x * cols;
  float* yr = y + (long long)blockIdx.x * cols;
  float m = -INFINITY;
  for (int j = threadIdx.x; j < cols; j += blockDim.x) m = fmaxf(m, xr[j]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  m = sh[0];
  for (int k = 1; k < (blockDim.x >> 5); ++k) m = fmaxf(m, sh[k]);
  __syncthreads();
  float s = 0.f;
  for (int j = threadIdx.x; j < cols; j += blockDim.x) {
    float e = expf(xr[j] - m);
    yr[j] = e;
    s += e;
  }
  s = block_sum(s, sh);
  float inv = 1.0f / s;
  for (int j = threadIdx.x; j < cols; j += blockDim.x) yr[j] *= inv;
}
__global__ void softmax_bwd_kernel(float* __restrict__ dx, const float* __restrict__ dy, const float* __restrict__ y, int cols) {
  __shared__ float sh[32];
  long long off = (long long)blockIdx.x * cols;
  float s = 0.f;
  for (int j = threadIdx.x; j < cols; j += blockDim.x) s += dy[off + j] * y[off + j];
  s = block_sum(s, sh);
  for (int j = threadIdx.x; j < cols; j += blockDim.x) dx[off + j] = y[off + j] * (dy[off + j] - s);
}
// Warp-per-row softmax for rows of up to 1024 columns (attention: 1024 keys): the row lives in registers (float4 x NV per
// lane), so forward reads and writes each element exactly once and backward reads dy, y once and writes dx once.
template <int NV>      // float4s per lane: cols == 128 * NV
__global__ void softmax_fwd_warp_kernel(float4* __restrict__ y, const float4* __restrict__ x, long long rows) {
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xr = x + row * (32 * NV);
  float4 v[NV];
  float m = -INFINITY;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i] = xr[i * 32 + lane];
    m = fmaxf(m, fmaxf(fmaxf(v[i].x, v[i].y), fmaxf(v[i].z, v[i].w)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x = expf(v[i].x - m); v[i].y = expf(v[i].y - m); v[i].z = expf(v[i].z - m); v[i].w = expf(v[i].w - m);
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
  s = warp_sum(s);
  float inv = 1.0f / s;
  float4* yr = y + row * (32 * NV);
#pragma unroll
  for (int i = 0; i < NV; ++i) yr[i * 32 + lane] = make_float4(v[i].x * inv, v[i].y * inv, v[i].z * inv, v[i].w * inv);
}
template <int NV>
__global__ void softmax_bwd_warp_kernel(float4* __restrict__ dx, const float4* __restrict__ dy, const float4* __restrict__ y,
                                        long long rows) {
  long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  long long off = row * (32 * NV);
  float4 g[NV], p[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    g[i] = dy[off + i * 32 + lane];
    p[i] = y[off + i * 32 + lane];
    s += (g[i].x * p[i].x + g[i].y * p[i].y) + (g[i].z * p[i].z + g[i].w * p[i].w);
  }
  s = warp_sum(s);
#pragma unroll
  for (int i = 0; i < NV; ++i)
    dx[off + i * 32 + lane] = make_float4(p[i].x * (g[i].x - s), p[i].y * (g[i].y - s), p[i].z * (g[i].z - s), p[i].w * (g[i].w - s));
}

// out[n, 2i+a, 2j+b, :] = bias for (a,b) != (0,0): the three bias-only sub-pixel phases of a 1x1 conv over a zero-inserted
// input (BigGAN's up-sampling shortcut, resnet_biggan.py:143-146)
__global__ void upsample1x1_bias_phases_kernel(float* __restrict__ out, const float* __restrict__ bias, int n, int oh, int ow, int c) {
  long long tot = (long long)n * oh * ow * c;
  EW_LOOP(i, tot) {
    int ch = (int)(i % c);
    long long t = i / c;
    int x = (int)(t % ow);
    int yy = (int)((t / ow) % oh);
    if ((x | yy) & 1) out[i] = bias ? bias[ch] : 0.f;
  }
}

__global__ void rowdot_kernel(float* __restrict__ out, const float* __restrict__ a, const float* __restrict__ b, long long rows, int cols) {
  long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  float s = 0.f;
  for (int j = lane; j < cols; j += 32) s += a[warp * cols + j] * b[warp * cols + j];
  s = warp_sum(s);
  if (lane == 0) out[warp] = s;
}
__global__ void rowscale_kernel(float* __restrict__ y, const float* __restrict__ a, const float* __restrict__ s, long long n, int cols) {
  EW_LOOP(i, n) y[i] = a[i] * s[i / cols];
}

// ---- losses: single block, b <= a few thousand logits
__device__ __forceinline__ float sce(float x, float z) { return fmaxf(x, 0.f) - x * z + log1pf(expf(-fabsf(x))); }

__global__ void gan_loss_kernel(int kind, const float* __restrict__ lr, const float* __restrict__ lf, int b, float* out4,
                                float* dl, int which) {
  __shared__ float sh[32];
  float sr = 0.f, sf = 0.f, sg = 0.f;
  float invb = 1.0f / (float)b;
  for (int i = threadIdx.x; i < b; i += blockDim.x) {
    float r = lr[i], f = lf[i];
    float dr = 0.f, df = 0.f;   // gradients wrt the real / fake logit of the requested loss
    if (kind == CGAN_LOSS_NON_SATURATING) {
      sr += sce(r, 1.f); sf += sce(f, 0.f); sg += sce(f, 1.f);
      float pr = sigmoidf_(r), pf = sigmoidf_(f);
      if (which == 0) { dr = (pr - 1.f) * invb; df = pf * invb; } else { df = (pf - 1.f) * invb; }
    } else if (kind == CGAN_LOSS_HINGE) {
      sr += fmaxf(1.f - r, 0.f); sf += fmaxf(1.f + f, 0.f); sg += -f;
      if (which == 0) { dr = (1.f - r > 0.f) ? -invb : 0.f; df = (1.f + f > 0.f) ? invb : 0.f; } else { df = -invb; }
    } else if (kind == CGAN_LOSS_WASSERSTEIN) {
      sr += -r; sf += f; sg += -f;
      if (which == 0) { dr = -invb; df = invb; } else { df = -invb; }
    } else {  // least squares on probabilities d = sigmoid(logit)
      float pr = sigmoidf_(r), pf = sigmoidf_(f);
      sr += (pr - 1.f) * (pr - 1.f); sf += pf * pf; sg += 0.5f * (pf - 1.f) * (pf - 1.f);
      if (which == 0) { dr = 0.5f * 2.f * (pr - 1.f) * pr * (1.f - pr) * invb; df = 0.5f * 2.f * pf * pf * (1.f - pf) * invb; }
      else { df = (pf - 1.f) * pf * (1.f - pf) * invb; }
    }
    if (dl) { dl[i] = dr; dl[b + i] = df; }
  }
  sr = block_sum(sr, sh);
  sf = block_sum(sf, sh);
  sg = block_sum(sg, sh);
  if (threadIdx.x == 0) {
    float a = sr * invb, c = sf * invb, g = sg * invb;
    float d = a + c;
    if (kind == CGAN_LOSS_LEAST_SQUARES) d = 0.5f * (a + c);
    out4[0] = d; out4[1] = a; out4[2] = c; out4[3] = g;
  }
}

// one block per sample: slope_n = sqrt(1e-4 + sum g^2)
__global__ void gp_slopes_kernel(float* slopes, const float* __restrict__ g, long long per) {
  __shared__ float sh[32];
  const float* p = g + (long long)blockIdx.x * per;
  float s = 0.f;
  for (long long i = threadIdx.x; i < per; i += blockDim.x) s += p[i] * p[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) slopes[blockIdx.x] = sqrtf(0.0001f + s);
}
__global__ void gp_penalty_kernel(float* pen, const float* slopes, int n) {
  __shared__ float sh[32];
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { float d = slopes[i] - 1.0f; s += d * d; }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) *pen = s / (float)n;
}
__global__ void gp_grad_kernel(float* __restrict__ dg, const float* __restrict__ g, const float* __restrict__ slopes,
                               long long per, long long tot, float coef) {
  EW_LOOP(i, tot) {
    float s = slopes[i / per];
    dg[i] = coef * (s - 1.0f) / s * g[i];
  }
}

__global__ void step_inc_kernel(int32_t* step) { *step += 1; }

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, float lr, float b1, float b2, float eps, float gscale, const int32_t* step,
                            float* __restrict__ ema, float ema_decay, int32_t ema_start) {
  int t = *step;   // already incremented
  // lr_t in double then rounded once, as the host-side TF kernel does
  double lr_t_d = (double)lr * sqrt(1.0 - pow((double)b2, (double)t)) / (1.0 - pow((double)b1, (double)t));
  float lr_t = (float)lr_t_d;
  float d = ((t - 1) >= ema_start) ? ema_decay : 0.0f;
  EW_LOOP(i, n) {
    float gi = g[i] * gscale;
    float mi = m[i] * b1 + (1.0f - b1) * gi;
    float vi = v[i] * b2 + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    float pi = p[i] - lr_t * mi / (sqrtf(vi) + eps);
    p[i] = pi;
    if (ema) { float e = ema[i]; ema[i] = e - (e - pi) * (1.0f - d); }
  }
}

}  // namespace

#define NONNULL(ctx) do { if (!(ctx)) return CGAN_ERR_ARG; } while (0)

int cgan_fill(cgan_ctx* ctx, float* d, float v, int64_t n) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, n >= 0 && (d || n == 0), "bad argument");
  if (n == 0) return CGAN_OK;
  fill_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(d, v, n);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_copy(cgan_ctx* ctx, float* d, const float* s, int64_t n) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, n >= 0 && ((d && s) || n == 0), "bad argument");
  if (n == 0) return CGAN_OK;
  copy_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(d, s, n);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_copy2d(cgan_ctx* ctx, float* d, int dld, int doff, const float* s, int sld, int soff, int64_t rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, d && s && rows >= 0 && cols >= 0 && doff >= 0 && soff >= 0, "bad argument");
  CGAN_REQUIRE(ctx, doff + cols <= dld && soff + cols <= sld, "column window exceeds leading dimension");
  if (rows * cols == 0) return CGAN_OK;
  copy2d_kernel<<<ew_grid(ctx, rows * cols), 256, 0, ctx->stream>>>(d, dld, doff, s, sld, soff, rows, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_axpby(cgan_ctx* ctx, float* y, float a, const float* x, float b, const float* y0, float c, int64_t n) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && n >= 0, "bad argument");
  if (n == 0) return CGAN_OK;
  axpby_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(y, a, x, b, y0, c, n);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_scale_by_dev(cgan_ctx* ctx, float* y, const float* x, const float* s, float mul, int inverse, int64_t n) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && s && n >= 0, "bad argument");
  if (n == 0) return CGAN_OK;
  scale_by_dev_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(y, x, s, mul, inverse, n);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_dot(cgan_ctx* ctx, float* out, const float* a, const float* b, int64_t n) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && a && b && n > 0, "bad argument");
  int blocks = ew_grid(ctx, n);
  if (blocks > 1024) blocks = 1024;
  void* ws = nullptr;
  int rc = cgan_ws(ctx, 1024 * sizeof(float), &ws);
  if (rc) return rc;
  float* part = reinterpret_cast<float*>(ws);
  dot_partial_kernel<<<blocks, 256, 0, ctx->stream>>>(part, a, b, n);
  CGAN_LAUNCHED(ctx);
  sum_final_kernel<<<1, 256, 0, ctx->stream>>>(out, part, blocks, 1.0f);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_interpolate(cgan_ctx* ctx, float* y, const float* x, const float* xf, const float* alpha, int n, int64_t per) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && xf && alpha && n > 0 && per > 0, "bad argument");
  long long tot = (long long)n * per;
  interpolate_kernel<<<ew_grid(ctx, tot), 256, 0, ctx->stream>>>(y, x, xf, alpha, per, tot);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_one_hot(cgan_ctx* ctx, float* out, const int32_t* labels, int n, int classes) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && labels && n > 0 && classes > 0, "bad argument");
  one_hot_kernel<<<ew_grid(ctx, (long long)n * classes), 256, 0, ctx->stream>>>(out, labels, n, classes);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_bias_add(cgan_ctx* ctx, float* y, const float* x, const float* bias, int64_t rows, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && bias && rows > 0 && c > 0, "bad argument");
  bias_add_kernel<<<ew_grid(ctx, rows * c), 256, 0, ctx->stream>>>(y, x, bias, rows * c, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_act_fwd(cgan_ctx* ctx, float* y, const float* x, int kind, float leak, int64_t n) {
  NONNULL(ctx);
  const int rnd = (kind & CGAN_ACT_ROUND_TF32) ? 1 : 0;
  kind &= ~CGAN_ACT_ROUND_TF32;
  CGAN_REQUIRE(ctx, y && x && n >= 0 && kind >= 1 && kind <= 4, "bad argument");
  if (n == 0) return CGAN_OK;
  act_fwd_kernel<<<ew_grid(ctx, (n + 3) / 4), 256, 0, ctx->stream>>>(y, x, kind, leak, n, rnd);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_act_bwd(cgan_ctx* ctx, float* dx, const float* dy, const float* ref, int kind, float leak, int64_t n) {
  NONNULL(ctx);
  const int rnd = (kind & CGAN_ACT_ROUND_TF32) ? 1 : 0;
  kind &= ~CGAN_ACT_ROUND_TF32;
  CGAN_REQUIRE(ctx, dx && dy && ref && n >= 0 && kind >= 1 && kind <= 4, "bad argument");
  if (n == 0) return CGAN_OK;
  act_bwd_kernel<<<ew_grid(ctx, (n + 3) / 4), 256, 0, ctx->stream>>>(dx, dy, ref, kind, leak, n, rnd);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_conv_post_epilogue(cgan_ctx* ctx, float* y, int64_t rows, int c, int ld, const float* residual, const float* mask,
                            float mask_leak, int relu, int round_out) {
  if (rows * c == 0) return CGAN_OK;
  conv_post_kernel<<<ew_grid(ctx, rows * c), 256, 0, ctx->stream>>>(y, rows, c, ld, residual, mask, mask_leak, relu, round_out);
  CGAN_LAUNCHED(ctx);
  return CGAN_OK;
}

namespace {
__global__ void random_uniform_kernel(float* __restrict__ out, long long n, unsigned long long seed, unsigned long long offset) {
  EW_LOOP(i, n) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (offset + (unsigned long long)i + 1ull);     // SplitMix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    out[i] = (float)(z >> 40) * (1.0f / 16777216.0f);
  }
}
}  // namespace

int cgan_random_uniform(cgan_ctx* ctx, float* out, int64_t n, uint64_t seed, uint64_t offset) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && n >= 0, "bad argument");
  if (n == 0) return CGAN_OK;
  random_uniform_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(out, n, seed, offset);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}

int cgan_rot90(cgan_ctx* ctx, float* y, const float* x, int n, int hw, int c, int k) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && n > 0 && hw > 0 && c > 0 && k >= 1 && k <= 3, "bad argument");
  rot90_kernel<<<ew_grid(ctx, (long long)n * hw * hw * c), 256, 0, ctx->stream>>>(y, x, n, hw, c, k);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_rotation_loss(cgan_ctx* ctx, float* loss_out, float* dlogits, const float* logits, int rows, int num_rotations) {
  NONNULL(ctx);
  CGAN_REQUIRE(ctx, loss_out && logits && rows > 0 && num_rotations > 0 && rows % num_rotations == 0, "rows must be a multiple of num_rotations");
  rotation_loss_kernel<<<1, 256, 0, ctx->stream>>>(loss_out, dlogits, logits, rows, num_rotations);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_row_has_label(cgan_ctx* ctx, float* out, const float* y, int rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && y && rows > 0 && cols > 0, "bad argument");
  row_has_label_kernel<<<ew_grid(ctx, rows), 256, 0, ctx->stream>>>(out, y, rows, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_argmax_one_hot(cgan_ctx* ctx, float* out, const float* logits, int rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && logits && rows > 0 && cols > 0, "bad argument");
  argmax_one_hot_kernel<<<ew_grid(ctx, rows), 256, 0, ctx->stream>>>(out, logits, rows, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_softmax_xent(cgan_ctx* ctx, float* loss_out, float* dlogits, const float* logits, const float* labels,
                      const float* weights, int rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, loss_out && logits && labels && rows > 0 && cols > 0, "bad argument");
  softmax_xent_kernel<<<1, 256, 0, ctx->stream>>>(loss_out, dlogits, logits, labels, weights, rows, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_add(cgan_ctx* ctx, float* y, const float* a, const float* b, int64_t n) { return cgan_add_tf32(ctx, y, a, b, n, 0); }
int cgan_add_tf32(cgan_ctx* ctx, float* y, const float* a, const float* b, int64_t n, int round_tf32) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && a && b && n >= 0, "bad argument");
  if (n == 0) return CGAN_OK;
  add_kernel<<<ew_grid(ctx, (n + 3) / 4), 256, 0, ctx->stream>>>(y, a, b, n, round_tf32 ? 1 : 0);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
#define POOL_ARGS_OK(ctx) CGAN_REQUIRE(ctx, n > 0 && h > 0 && w > 0 && c > 0 && h % 2 == 0 && w % 2 == 0, "need even h,w")
int cgan_avgpool2_fwd(cgan_ctx* ctx, float* y, const float* x, int n, int h, int w, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x, "null pointer"); POOL_ARGS_OK(ctx);
  if (c % 4 == 0 && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x)) & 15) == 0)
    avgpool2_fwd_v4_kernel<<<ew_grid(ctx, (long long)n * h * w * c / 16), 256, 0, ctx->stream>>>(
        reinterpret_cast<float4*>(y), reinterpret_cast<const float4*>(x), n, h, w, c / 4);
  else
    avgpool2_fwd_kernel<<<ew_grid(ctx, (long long)n * h * w * c / 4), 256, 0, ctx->stream>>>(y, x, n, h, w, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_avgpool2_bwd(cgan_ctx* ctx, float* dx, const float* dy, int n, int h, int w, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, dx && dy, "null pointer"); POOL_ARGS_OK(ctx);
  if (c % 4 == 0 && ((reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dy)) & 15) == 0)
    avgpool2_bwd_v4_kernel<<<ew_grid(ctx, (long long)n * h * w * c / 16), 256, 0, ctx->stream>>>(
        reinterpret_cast<float4*>(dx), reinterpret_cast<const float4*>(dy), n, h, w, c / 4);
  else
    avgpool2_bwd_kernel<<<ew_grid(ctx, (long long)n * h * w * c), 256, 0, ctx->stream>>>(dx, dy, n, h, w, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_maxpool2_fwd(cgan_ctx* ctx, float* y, const float* x, int n, int h, int w, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x, "null pointer"); POOL_ARGS_OK(ctx);
  maxpool2_fwd_kernel<<<ew_grid(ctx, (long long)n * h * w * c / 4), 256, 0, ctx->stream>>>(y, x, n, h, w, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_maxpool2_bwd(cgan_ctx* ctx, float* dx, const float* dy, const float* x, int n, int h, int w, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, dx && dy && x, "null pointer"); POOL_ARGS_OK(ctx);
  maxpool2_bwd_kernel<<<ew_grid(ctx, (long long)n * h * w * c / 4), 256, 0, ctx->stream>>>(dx, dy, x, n, h, w, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_pool2d_fwd(cgan_ctx* ctx, float* y, const float* x, int n, int h, int w, int c, int k, int stride, int pad_t,
                    int pad_l, int oh, int ow, int mode) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && n > 0 && h > 0 && w > 0 && c > 0 && k > 0 && stride > 0 && oh > 0 && ow > 0, "bad argument");
  CGAN_REQUIRE(ctx, mode == 0 || mode == 1, "mode must be 0 (max) or 1 (avg)");
  if (c % 4 == 0 && ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x)) & 15) == 0)
    pool2d_fwd_v4_kernel<<<ew_grid(ctx, (long long)n * oh * ow * c / 4), 256, 0, ctx->stream>>>(
        reinterpret_cast<float4*>(y), reinterpret_cast<const float4*>(x), n, h, w, c / 4, k, stride, pad_t, pad_l, oh, ow, mode);
  else
    pool2d_fwd_kernel<<<ew_grid(ctx, (long long)n * oh * ow * c), 256, 0, ctx->stream>>>(y, x, n, h, w, c, k, stride, pad_t, pad_l,
                                                                                      oh, ow, mode);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_globalpool_fwd(cgan_ctx* ctx, float* y, const float* x, int n, int hw, int c, float scale) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && n > 0 && hw > 0 && c > 0, "bad argument");
  globalpool_fwd_kernel<<<ew_grid(ctx, (long long)n * c), 256, 0, ctx->stream>>>(y, x, n, hw, c, scale);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_globalpool_bwd(cgan_ctx* ctx, float* dx, const float* dy, int n, int hw, int c, float scale) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, dx && dy && n > 0 && hw > 0 && c > 0, "bad argument");
  globalpool_bwd_kernel<<<ew_grid(ctx, (long long)n * hw * c), 256, 0, ctx->stream>>>(dx, dy, n, hw, c, scale);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_softmax_fwd(cgan_ctx* ctx, float* y, const float* x, int64_t rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && x && rows > 0 && cols > 0 && rows < (1ll << 31), "bad argument");
  const bool al = ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(x)) & 15) == 0;
  const unsigned wblocks = (unsigned)((rows * 32 + 255) / 256);
  if (al && cols == 1024)
    softmax_fwd_warp_kernel<8><<<wblocks, 256, 0, ctx->stream>>>(reinterpret_cast<float4*>(y), reinterpret_cast<const float4*>(x), rows);
  else if (al && cols == 256)
    softmax_fwd_warp_kernel<2><<<wblocks, 256, 0, ctx->stream>>>(reinterpret_cast<float4*>(y), reinterpret_cast<const float4*>(x), rows);
  else
    softmax_fwd_kernel<<<(unsigned)rows, 256, 0, ctx->stream>>>(y, x, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_softmax_bwd(cgan_ctx* ctx, float* dx, const float* dy, const float* y, int64_t rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, dx && dy && y && rows > 0 && cols > 0 && rows < (1ll << 31), "bad argument");
  const bool al = ((reinterpret_cast<uintptr_t>(dx) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  const unsigned wblocks = (unsigned)((rows * 32 + 255) / 256);
  if (al && cols == 1024)
    softmax_bwd_warp_kernel<8><<<wblocks, 256, 0, ctx->stream>>>(reinterpret_cast<float4*>(dx), reinterpret_cast<const float4*>(dy),
                                                                 reinterpret_cast<const float4*>(y), rows);
  else if (al && cols == 256)
    softmax_bwd_warp_kernel<2><<<wblocks, 256, 0, ctx->stream>>>(reinterpret_cast<float4*>(dx), reinterpret_cast<const float4*>(dy),
                                                                 reinterpret_cast<const float4*>(y), rows);
  else
    softmax_bwd_kernel<<<(unsigned)rows, 256, 0, ctx->stream>>>(dx, dy, y, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_upsample1x1_bias_phases(cgan_ctx* ctx, float* out, const float* bias, int n, int oh, int ow, int c) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && n > 0 && oh > 0 && ow > 0 && c > 0, "bad argument");
  upsample1x1_bias_phases_kernel<<<ew_grid(ctx, (long long)n * oh * ow * c), 256, 0, ctx->stream>>>(out, bias, n, oh, ow, c);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_rowdot(cgan_ctx* ctx, float* out, const float* a, const float* b, int64_t rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, out && a && b && rows > 0 && cols > 0, "bad argument");
  rowdot_kernel<<<cdiv(rows * 32, 256), 256, 0, ctx->stream>>>(out, a, b, rows, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_rowscale(cgan_ctx* ctx, float* y, const float* a, const float* s, int64_t rows, int cols) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, y && a && s && rows > 0 && cols > 0, "bad argument");
  rowscale_kernel<<<ew_grid(ctx, rows * cols), 256, 0, ctx->stream>>>(y, a, s, rows * cols, cols);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_gan_loss(cgan_ctx* ctx, int kind, const float* lr, const float* lf, int b, float* out4, float* dl, int which) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, lr && lf && out4 && b > 0 && kind >= 0 && kind <= 3 && (which == 0 || which == 1), "bad argument");
  gan_loss_kernel<<<1, 256, 0, ctx->stream>>>(kind, lr, lf, b, out4, dl, which);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
int cgan_gp_penalty(cgan_ctx* ctx, float* pen, float* dg, const float* g, int n, int64_t per, float weight) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, pen && g && n > 0 && per > 0, "bad argument");
  void* ws = nullptr;
  int rc = cgan_ws(ctx, (size_t)n * sizeof(float), &ws);
  if (rc) return rc;
  float* slopes = reinterpret_cast<float*>(ws);
  gp_slopes_kernel<<<n, 256, 0, ctx->stream>>>(slopes, g, per);
  CGAN_LAUNCHED(ctx);
  gp_penalty_kernel<<<1, 256, 0, ctx->stream>>>(pen, slopes, n);
  CGAN_LAUNCHED(ctx);
  if (dg) {
    long long tot = (long long)n * per;
    gp_grad_kernel<<<ew_grid(ctx, tot), 256, 0, ctx->stream>>>(dg, g, slopes, per, tot, 2.0f * weight / (float)n);
    CGAN_LAUNCHED(ctx);
  }
  return CGAN_OK;
}
int cgan_adam_step(cgan_ctx* ctx, float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2,
                   float eps, float gscale, int32_t* step, float* ema, float ema_decay, int32_t ema_start) {
  NONNULL(ctx); CGAN_REQUIRE(ctx, p && g && m && v && step && n > 0, "bad argument");
  step_inc_kernel<<<1, 1, 0, ctx->stream>>>(step);
  CGAN_LAUNCHED(ctx);
  adam_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(p, g, m, v, n, lr, b1, b2, eps, gscale, step, ema, ema_decay, ema_start);
  CGAN_LAUNCHED(ctx); return CGAN_OK;
}
