// Shared helpers for the sm_100a kernels behind include/cgan_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/cgan_b200.h"

struct cgan_ctx {
  int device;
  cudaStream_t stream;
  void* ws;
  size_t ws_bytes;
  int math_mode;
  int64_t launches;
  int num_sms;
  int tc_mt_max;       // tcgen05 kernels: max tiles per CTA sharing one operand tile (CGAN_OPT_TC_MT, default 2)
  int tc_halo;         // 3x3 stride-1 tcgen05 convolutions use the halo variant (CGAN_OPT_TC_HALO, default 1)
  int tc_thin;         // image-side (<= 4 channel) convolutions through 32-wide patch tensors on tcgen05 (CGAN_OPT_TC_THIN, default 1)
  int last_path;       // CGAN_PATH_* of the most recent contraction (cgan_ctx_get_option(CGAN_OPT_LAST_PATH))
  unsigned* counters;  // CGAN_NUM_COUNTERS zero-initialised tickets for single-launch two-stage reductions (norm.cu)
  void* p2p;           // peer-memory all-reduce state (p2p.cu), null until cgan_p2p_local_handle
  char err[512];
};

constexpr int CGAN_NUM_COUNTERS = 1 << 18;

static inline int cgan_fail(cgan_ctx* ctx, int code, const char* fmt, const char* a = "", const char* b = "") {
  if (ctx) snprintf(ctx->err, sizeof(ctx->err), fmt, a, b);
  return code;
}

#define CGAN_REQUIRE(ctx, cond, msg)                                              \
  do {                                                                            \
    if (!(cond)) return cgan_fail((ctx), CGAN_ERR_ARG, "%s: %s", __func__, msg);  \
  } while (0)

#define CGAN_CUDA(ctx, call)                                                                        \
  do {                                                                                              \
    cudaError_t e__ = (call);                                                                       \
    if (e__ != cudaSuccess) return cgan_fail((ctx), CGAN_ERR_CUDA, "%s: %s", __func__, cudaGetErrorString(e__)); \
  } while (0)

// after every kernel launch: count it and surface launch-configuration errors without synchronising
#define CGAN_LAUNCHED(ctx)                                                                          \
  do {                                                                                              \
    (ctx)->launches++;                                                                              \
    cudaError_t e__ = cudaGetLastError();                                                           \
    if (e__ != cudaSuccess) return cgan_fail((ctx), CGAN_ERR_CUDA, "%s: launch: %s", __func__, cudaGetErrorString(e__)); \
  } while (0)

// Workspace owned by the context; grows on demand outside stream capture only.
static inline int cgan_ws(cgan_ctx* ctx, size_t bytes, void** out) {
  if (bytes > ctx->ws_bytes) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(ctx->stream, &st);
    if (st != cudaStreamCaptureStatusNone)
      return cgan_fail(ctx, CGAN_ERR_WORKSPACE, "%s: workspace would grow during stream capture (warm up first)%s", "cgan_ws");
    size_t want = bytes + bytes / 4 + (1 << 20);
    want = (want + 255) / 256 * 256;
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess && ctx->ws) e = cudaFree(ctx->ws);
    ctx->ws = nullptr;
    ctx->ws_bytes = 0;
    if (e == cudaSuccess) e = cudaMalloc(&ctx->ws, want);
    if (e != cudaSuccess) return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: %s", "cgan_ws", cudaGetErrorString(e));
    ctx->ws_bytes = want;
  }
  *out = ctx->ws;
  return CGAN_OK;
}

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum; result valid in all threads. `sh` must hold 32 floats.
__device__ __forceinline__ float block_sum(float v, float* sh) {
  int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) sh[w] = v;
  __syncthreads();
  int nw = (blockDim.x + 31) >> 5;
  float r = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.f;
  if (w == 0) {
    r = warp_sum(r);
    if (lane == 0) sh[0] = r;
  }
  __syncthreads();
  r = sh[0];
  return r;
}

// Optional arguments of the tcgen05 convolution launcher cgan_conv_tc (all zero = the plain convolution)
struct TcExtra {
  const float* wprep;       // weights already prepared by cgan_tc_prep_weights (shared by several launches)
  int a_prerounded;         // the activation operand already holds TF32-representable values: skip the in-smem rounding
  int round_out;            // store TF32-rounded outputs
  const float* residual;    // + residual (output geometry), before the activation
  const float* mask;        // (leaky-)ReLU backward fused into the epilogue: out = mask > 0 ? v : mask_leak * v
  float mask_leak;
  int nphases;              // > 1: several sub-pixel phases in one launch (tap list = concatenation, see cgan_conv_tc)
  int ph_tap0[5];
  long long ph_base[4];
};

// internal (C++ linkage) entry points shared between translation units
int cgan_conv2d_fwd_simt(cgan_ctx*, const cgan_conv_desc*, const float* x, const float* w, const float* bias, float* y,
                         int relu, int ldy);
int cgan_conv2d_dgrad_simt(cgan_ctx*, const cgan_conv_desc*, const float* dy, const float* w, float* dx);
int cgan_conv_post_epilogue(cgan_ctx* ctx, float* y, int64_t rows, int c, int ld, const float* residual, const float* mask,
                            float mask_leak, int relu, int round_out);
int cgan_upsample1x1_bias_phases(cgan_ctx* ctx, float* out, const float* bias, int n, int oh, int ow, int c);
int cgan_gemm_batched_simt(cgan_ctx* ctx, int ta, int tb, int m, int n, int k, float alpha, const float* a, int lda,
                           int64_t sa, const float* b, int ldb, int64_t sb, float beta, float* c, int ldc, int64_t sc, int batch);
