// Fused self-attention of the non-local block (arch_ops.py:734-753) on tcgen05 — math_mode 1.
//
//   O[i] = softmax(Q[i] K[i]^T) V[i]          Q = theta [Lq, dk], K = phi [Lk, dk], V = g [Lk, dv] per image i
//
// The reference materialises the [Lq, Lk] score matrix (tf.matmul -> tf.nn.softmax -> tf.matmul); at BigGAN-128 that is
// 4096 x 1024 floats per image, 4.3 GB per batch of 256, crossing HBM three times per direction.  Here the scores never
// leave the SM — not even the tensor memory: S tiles are produced by tcgen05.mma into TMEM, read by the softmax warps with
// tcgen05.ld, exponentiated, rounded to TF32 and written back IN PLACE with tcgen05.st, and the second tcgen05.mma takes them
// as its A operand straight from TMEM (no shared-memory tile, no generic -> async proxy fence on the per-tile chain).
//
// Operand tiles stream through multi-stage shared-memory rings filled by ONE polling TMA thread, which never blocks on one
// ring while another could be refilled (measured history of the variants: DESIGN.md section 7, profiles/r2_attention_*.txt).
// Forward (attn_fwd_kernel): one CTA per 128 queries of one image, key tiles of 64.
//   pass 1: S_j = Q K_j^T (M=128, N=64, K=8 per MMA, dk <= 32 zero-padded by TMA) -> row maxima m.
//   pass 2: S_j again (K has 4x fewer channels than V: recomputing costs 1/4 of the P V MMAs and avoids rescaling O in
//           TMEM), p = exp(s - m), l += p, P -> TMEM (in place), O += P V_j (V is MN-major as it lies in HBM: the filter-gradient
//           kernel's SWIZZLE_128B_BASE32B operand form).  Epilogue: O / l, lse = m + log l (kept for the backward).
// Backward: P is recomputed from Q, K and lse (no [Lq, Lk] tensor is ever stored); with D = rowsum(dO * O),
//   dS = P * (dO V^T - D),  dQ = dS K,  dK = dS^T Q,  dV = P^T dO.
//   attn_bwd_dq_kernel: one CTA per 128 queries, loops over key tiles (accumulates dQ in TMEM);
//   attn_bwd_dkv_kernel: one CTA per 128 keys, loops over query tiles of 64 (accumulates dK, dV in TMEM) — S^T and dP^T
//   are produced directly (M = keys), so no transposition pass exists and the summation order is fixed (deterministic).
// Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..9 = softmax / epilogue:
// TMEM lane quarter = warp % 4, two warps per quarter, each owning one 32-column half of every 64-column score tile.
//
// Operands are consumed as TF32: callers pass tensors already rounded to the nearest TF32 value (cgan_round_tf32 or a
// producer's ROUND_OUT epilogue); P and dS are rounded to nearest by the softmax warps.  Accumulation is fp32 in TMEM.
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int AT_THREADS = 320;
constexpr int AT_SWARPS = 8;         // softmax warps
constexpr int AT_TQ = 128;          // rows per CTA (UMMA M)
constexpr int AT_TK = 64;           // columns per score tile (UMMA N of the score MMAs)
constexpr float AT_LOG2E = 1.4426950408889634f;

constexpr int AT_MAX_STAGES = 4;
constexpr size_t AT_SMEM_MAX = 227 * 1024;

struct AtParams {
  int lq, lk, dk, dv;
  int ns_a, ns_b;       // ring depths: fwd K / V tiles; dq: key-tile ring (both operand groups); dkv: K-major / MN-major query groups
  int kq;               // MMA k-steps of the score contraction: ceil(dk / 8)
  int kv;               // MMA k-steps of a contraction over dv: ceil(dv / 8)
  int vg;               // 32-channel groups of V / dO: ceil(dv / 32)
  int nv;               // UMMA N of the contractions producing dv columns (dv, a multiple of 16)
  float* out;           // fwd: O          dq: dQ        dkv: dK
  float* out2;          // fwd: lse        dq: -         dkv: dV
  const float* lse;     // bwd
  const float* dsum;    // bwd: D = rowsum(dO * O)
};

// K-major, 128B-swizzled operand (rows x 32 fp32 = 128 B per row, 8-row groups 1024 B apart) — as conv_tc.cu
__device__ __forceinline__ uint64_t desc_k(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// MN-major 32-bit operand, SWIZZLE_128B_BASE32B: 32-channel groups 4096 B apart (LBO), 4-row groups 512 B apart (SBO) — as
// wgrad_tc.cu
__device__ __forceinline__ uint64_t desc_mn(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(4096 >> 4) << 16;
  d |= (uint64_t)(512 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;
  return d;
}
// instruction descriptor: D = F32, A = B = TF32, M = 128, N = n; b_mn: B operand MN-major
__device__ __forceinline__ uint32_t idesc(int n, int b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)b_mn << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(AT_TQ >> 4) << 24);
}

// mbarrier wait that traps instead of hanging the device if a protocol error ever leaves a barrier incomplete
__device__ __forceinline__ void bwait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  const long long t0 = clock64();
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
    if (ok) return;
    if (clock64() - t0 > 4000000000ll) __trap();
  }
}

// non-blocking probe (the TMA producer polls several rings: it must never block on one while another could be refilled)
__device__ __forceinline__ bool btest(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// the idle branch of a polling producer: back off briefly, trap after ~2 s without progress
__device__ __forceinline__ void poll_idle(long long& t_last) {
  __nanosleep(64);
  if (clock64() - t_last > 4000000000ll) __trap();
}

// round to the nearest TF32 value, ties away from zero — bit-identical to cvt.rna.tf32.f32 for finite values below the
// largest TF32 binade (probabilities and their products here), but two full-rate integer ops instead of one instruction on
// the quarter-rate conversion pipe, which the exponentials already saturate (ncu r2: softmax warps XU-bound)
__device__ __forceinline__ float rnd_tf32(float x) {
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}
__device__ __forceinline__ void fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void softmax_bar() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

// tcgen05.st 32 lanes x 32 columns: every thread writes 32 consecutive fp32 columns of ITS TMEM lane (the probabilities /
// dS go back where the scores came from: the next tcgen05.mma reads them as its A operand straight from TMEM)
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]),
        "f"(v[10]), "f"(v[11]), "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15]), "f"(v[16]), "f"(v[17]), "f"(v[18]), "f"(v[19]),
        "f"(v[20]), "f"(v[21]), "f"(v[22]), "f"(v[23]), "f"(v[24]), "f"(v[25]), "f"(v[26]), "f"(v[27]), "f"(v[28]), "f"(v[29]),
        "f"(v[30]), "f"(v[31]) : "memory");
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// D[tmem] (+)= A[tmem: 128 lanes x 8 fp32 columns per K step] * B[smem descriptor]
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

// one row of `dst` from the accumulator columns [0, ncols) at `taddr`, scaled; this thread takes the 32-column chunks
// c_begin, c_begin + c_step, ...
__device__ __forceinline__ void store_acc_row(float* dst, uint32_t taddr, int ncols, float scale, int c_begin, int c_step) {
  for (int c0 = c_begin * 32; c0 < ncols; c0 += c_step * 32) {
    uint32_t r[32];
    tmem_ld32(taddr + (uint32_t)c0, r);
#pragma unroll
    for (int j = 0; j < 32; j += 4)
      if (c0 + j < ncols)
        *reinterpret_cast<float4*>(dst + c0 + j) = make_float4(__uint_as_float(r[j]) * scale, __uint_as_float(r[j + 1]) * scale,
                                                                __uint_as_float(r[j + 2]) * scale, __uint_as_float(r[j + 3]) * scale);
  }
}

// ------------------------------------------------------------------------------------------------------------ forward
// shared memory: Q 16 KB | K ring ns_a x 8 KB | V ring ns_b x (vg x 8 KB) | barriers | row max / sum exchange.
// TMEM (256 columns): S0 / P0 @0, S1 / P1 @64, O @128.
__global__ void __launch_bounds__(AT_THREADS, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                const __grid_constant__ CUtensorMap tm_v, const AtParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int v_bytes = p.vg * 2 * 4096;
  uint8_t* sQ = smem;
  uint8_t* sK = smem + 16384;
  uint8_t* sV = sK + p.ns_a * 8192;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sV + p.ns_b * v_bytes);
  uint64_t* q_full = bars;                          // 1
  uint64_t* k_full = bars + 1;                      // AT_MAX_STAGES
  uint64_t* k_empty = k_full + AT_MAX_STAGES;
  uint64_t* v_full = k_empty + AT_MAX_STAGES;
  uint64_t* v_empty = v_full + AT_MAX_STAGES;
  uint64_t* s_full = v_empty + AT_MAX_STAGES;       // 2: scores of a tile are in TMEM
  uint64_t* s_empty = s_full + 2;                   // 2: pass 1 — the softmax warps have read them
  uint64_t* p_ready = s_empty + 2;                  // 2: pass 2 — the probabilities are back in TMEM
  uint64_t* pv_done = p_ready + 2;                  // 2: pass 2 — P V retired: the buffer may take new scores
  uint64_t* o_full = pv_done + 2;                   // 26 barriers
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(o_full + 1);
  float* sX = reinterpret_cast<float*>(bars + 32);       // [2][128]: row maxima / row sums of the two column halves

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * AT_TQ, img = blockIdx.y;
  const int nkt = p.lk / AT_TK;                     // even (lk is a multiple of 128): tile parity == buffer in both passes

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_q) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_k) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_v) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      mbar_init(q_full, 1);
      for (int s = 0; s < AT_MAX_STAGES; ++s) {
        mbar_init(&k_full[s], 1); mbar_init(&k_empty[s], 1); mbar_init(&v_full[s], 1); mbar_init(&v_empty[s], 1);
      }
      for (int s = 0; s < 2; ++s) {
        mbar_init(&s_full[s], 1); mbar_init(&s_empty[s], AT_SWARPS); mbar_init(&p_ready[s], AT_SWARPS); mbar_init(&pv_done[s], 1);
      }
      mbar_init(o_full, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc(tmem_ptr, 256);
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(q_full, 16384);
      tma_load_4d(sQ, &tm_q, q_full, 0, q0, 0, img);
      // K tiles are consumed twice (pass 1: row maxima, pass 2), V tiles once; both rings are refilled as soon as a stage
      // drains, so V runs ns_b tiles ahead of pass 2 (its first tiles load during pass 1)
      int kt = 0, vt = 0;
      long long t_last = clock64();
      while (kt < 2 * nkt || vt < nkt) {
        bool progress = false;
        if (kt < 2 * nkt) {
          const int s = kt % p.ns_a;
          if (btest(&k_empty[s], ((kt / p.ns_a) & 1) ^ 1)) {
            mbar_expect_tx(&k_full[s], 8192);
            tma_load_4d(sK + s * 8192, &tm_k, &k_full[s], 0, (kt % nkt) * AT_TK, 0, img);
            ++kt; progress = true;
          }
        }
        if (vt < nkt) {
          const int s = vt % p.ns_b;
          if (btest(&v_empty[s], ((vt / p.ns_b) & 1) ^ 1)) {
            mbar_expect_tx(&v_full[s], (uint32_t)v_bytes);
            for (int kb = 0; kb < 2; ++kb)
              for (int g = 0; g < p.vg; ++g)
                tma_load_4d(sV + s * v_bytes + (kb * p.vg + g) * 4096, &tm_v, &v_full[s], g * 32, vt * AT_TK + kb * 32, 0, img);
            ++vt; progress = true;
          }
        }
        if (progress) t_last = clock64(); else poll_idle(t_last);
      }
    }
  } else if (warp == 1) {
    const uint32_t id_s = idesc(AT_TK, 0), id_pv = idesc(p.nv, 1);
    const uint32_t aQ = smem_u32(sQ), aK = smem_u32(sK), aV = smem_u32(sV);
    bwait(q_full, 0);
    // scores of tile `it` (0 .. 2 nkt - 1) into buffer it & 1.  The buffer's previous tenant is tile it - 2: in pass 1 it is
    // free once the softmax warps have read it (s_empty), in pass 2 once the P V product that reads it has retired (pv_done)
    auto issue_s = [&](int it) {
      const int ks = it % p.ns_a, sb = it & 1;
      bwait(&k_full[ks], (it / p.ns_a) & 1);
      if (it >= 2) {
        if (it - 2 < nkt) bwait(&s_empty[sb], ((it - 2) >> 1) & 1);
        else bwait(&pv_done[sb], ((it - 2 - nkt) >> 1) & 1);
      }
      fence_after();
      if (lane == 0) {
        for (int k = 0; k < p.kq; ++k)
          umma_tf32(tmem + (uint32_t)(sb * AT_TK), desc_k(aQ + k * 32), desc_k(aK + ks * 8192 + k * 32), id_s, k ? 1u : 0u);
        umma_commit(&k_empty[ks]);
        umma_commit(&s_full[sb]);
      }
      __syncwarp();
    };
    for (int it = 0; it < nkt; ++it) issue_s(it);          // pass 1: scores for the row maxima
    issue_s(nkt);
    for (int j = 0; j < nkt; ++j) {
      if (j + 1 < nkt) issue_s(nkt + j + 1);
      const int vs = j % p.ns_b, sb = j & 1;
      bwait(&p_ready[sb], (j >> 1) & 1);
      bwait(&v_full[vs], (j / p.ns_b) & 1);
      fence_after();
      if (lane == 0) {
        for (int kk = 0; kk < AT_TK / 8; ++kk)           // A = P from TMEM: 8 fp32 columns per K step
          umma_tf32_ts(tmem + 128, tmem + (uint32_t)(sb * AT_TK + kk * 8),
                       desc_mn(aV + vs * v_bytes + (kk >> 2) * p.vg * 4096 + (kk & 3) * 1024), id_pv, (j | kk) ? 1u : 0u);
        umma_commit(&pv_done[sb]);
        umma_commit(&v_empty[vs]);
        if (j == nkt - 1) umma_commit(o_full);
      }
      __syncwarp();
    }
  } else {
    const int quarter = warp & 3, half = (warp - 2) >> 2, row = quarter * 32 + lane;
    const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 32);
    float m = -INFINITY;
    for (int it = 0; it < nkt; ++it) {
      const int s = it & 1;
      bwait(&s_full[s], (it >> 1) & 1);
      fence_after();
      uint32_t r[32];
      tmem_ld32(tl + (uint32_t)(s * AT_TK), r);
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&s_empty[s]);
#pragma unroll
      for (int i = 0; i < 32; ++i) m = fmaxf(m, __uint_as_float(r[i]));
    }
    sX[half * 128 + row] = m;
    softmax_bar();
    m = fmaxf(sX[row], sX[128 + row]);
    softmax_bar();                       // sX is reused for the row sums
    const float m2 = m * AT_LOG2E;
    float l = 0.f;
    for (int j = 0; j < nkt; ++j) {
      const int it = nkt + j, s = it & 1;
      bwait(&s_full[s], (it >> 1) & 1);
      fence_after();
      uint32_t r[32];
      tmem_ld32(tl + (uint32_t)(s * AT_TK), r);
      float pv[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) { pv[i] = rnd_tf32(ex2(fmaf(__uint_as_float(r[i]), AT_LOG2E, -m2))); l += pv[i]; }
      tmem_st32(tl + (uint32_t)(s * AT_TK), pv);           // in place: the probabilities replace the scores
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_ready[s]);
    }
    sX[half * 128 + row] = l;
    softmax_bar();
    l = sX[row] + sX[128 + row];
    bwait(o_full, 0);
    fence_after();
    const long long grow = (long long)img * p.lq + q0 + row;
    store_acc_row(p.out + grow * p.dv, tmem + ((uint32_t)(quarter * 32) << 16) + 128, p.dv, 1.0f / l, half, 2);
    if (half == 0) p.out2[grow] = m + logf(l);
    fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    fence_after();
    tmem_dealloc(tmem, 256);
  }
}

// -------------------------------------------------------------------------------------------------------- backward: dQ
// shared memory: Q 16 KB | dO vg x 16 KB | key-tile ring ns_a x [K (K-major) 8 KB | V (K-major) vg x 8 KB | K (MN-major) 8 KB] |
// barriers.  TMEM (512 columns): buffer b @ b*128: S -> dS @+0, dP @+64; dQ @256.
__global__ void __launch_bounds__(AT_THREADS, 1)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_do,
                   const __grid_constant__ CUtensorMap tm_k, const __grid_constant__ CUtensorMap tm_vk,
                   const __grid_constant__ CUtensorMap tm_km, const AtParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = 16384 + p.vg * 8192;     // [K K-major 8 KB | V K-major vg x 8 KB | K MN-major 8 KB]
  uint8_t* sQ = smem;
  uint8_t* sdO = sQ + 16384;
  uint8_t* ring = sdO + p.vg * 16384;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ring + p.ns_a * stage_bytes);
  uint64_t* q_full = bars;
  uint64_t* km_full = bars + 1;                     // AT_MAX_STAGES each
  uint64_t* km_empty = km_full + AT_MAX_STAGES;
  uint64_t* mn_full = km_empty + AT_MAX_STAGES;
  uint64_t* mn_empty = mn_full + AT_MAX_STAGES;
  uint64_t* sd_full = mn_empty + AT_MAX_STAGES;     // 2: S and dP of a tile are in TMEM
  uint64_t* ds_ready = sd_full + 2;                 // 2: dS is back in TMEM
  uint64_t* dq_done = ds_ready + 2;                 // 2: dQ += dS K retired: the buffer may take the next tile
  uint64_t* dq_full = dq_done + 2;                  // 24 barriers
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(dq_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * AT_TQ, img = blockIdx.y;
  const int nkt = p.lk / AT_TK;

  if (warp == 1) {
    if (lane == 0) {
      mbar_init(q_full, 1);
      for (int s = 0; s < AT_MAX_STAGES; ++s) {
        mbar_init(&km_full[s], 1); mbar_init(&km_empty[s], 1); mbar_init(&mn_full[s], 1); mbar_init(&mn_empty[s], 1);
      }
      for (int s = 0; s < 2; ++s) { mbar_init(&sd_full[s], 1); mbar_init(&ds_ready[s], AT_SWARPS); mbar_init(&dq_done[s], 1); }
      mbar_init(dq_full, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc(tmem_ptr, 512);
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(q_full, (uint32_t)(16384 + p.vg * 16384));
      tma_load_4d(sQ, &tm_q, q_full, 0, q0, 0, img);
      for (int g = 0; g < p.vg; ++g) tma_load_4d(sdO + g * 16384, &tm_do, q_full, g * 32, q0, 0, img);
      // two operand groups per key tile with different lifetimes: the K-major K / V tiles are free once S and dP are
      // computed, the MN-major K tile once dQ has consumed dS
      int kt = 0, mt = 0;
      long long t_last = clock64();
      while (kt < nkt || mt < nkt) {
        bool progress = false;
        if (kt < nkt) {
          const int s = kt % p.ns_a;
          if (btest(&km_empty[s], ((kt / p.ns_a) & 1) ^ 1)) {
            uint8_t* st = ring + s * stage_bytes;
            mbar_expect_tx(&km_full[s], (uint32_t)(8192 + p.vg * 8192));
            tma_load_4d(st, &tm_k, &km_full[s], 0, kt * AT_TK, 0, img);
            for (int g = 0; g < p.vg; ++g) tma_load_4d(st + 8192 + g * 8192, &tm_vk, &km_full[s], g * 32, kt * AT_TK, 0, img);
            ++kt; progress = true;
          }
        }
        if (mt < nkt) {
          const int s = mt % p.ns_a;
          if (btest(&mn_empty[s], ((mt / p.ns_a) & 1) ^ 1)) {
            uint8_t* st = ring + s * stage_bytes + 8192 + p.vg * 8192;
            mbar_expect_tx(&mn_full[s], 8192);
            for (int kb = 0; kb < 2; ++kb) tma_load_4d(st + kb * 4096, &tm_km, &mn_full[s], 0, mt * AT_TK + kb * 32, 0, img);
            ++mt; progress = true;
          }
        }
        if (progress) t_last = clock64(); else poll_idle(t_last);
      }
    }
  } else if (warp == 1) {
    const uint32_t id_s = idesc(AT_TK, 0), id_dq = idesc(32, 1);
    const uint32_t aQ = smem_u32(sQ), adO = smem_u32(sdO), aR = smem_u32(ring);
    bwait(q_full, 0);
    auto issue_sd = [&](int j) {
      const int b = j & 1, s = j % p.ns_a;
      const uint32_t aKk = aR + s * stage_bytes, aVk = aKk + 8192;
      bwait(&km_full[s], (j / p.ns_a) & 1);
      if (j >= 2) bwait(&dq_done[b], ((j - 2) >> 1) & 1);        // the buffer's previous tile has been consumed by its dQ product
      fence_after();
      if (lane == 0) {
        // the two products accumulate into different TMEM columns: their MMAs are issued alternately so that consecutive
        // instructions in the tensor pipe do not depend on each other (a K step of N = 64 is 32 clk of math, far less than
        // the latency of a dependent accumulation)
        for (int kk = 0; kk < p.kv; ++kk) {
          umma_tf32(tmem + (uint32_t)(b * 128 + 64), desc_k(adO + (kk >> 2) * 16384 + (kk & 3) * 32),
                    desc_k(aVk + (kk >> 2) * 8192 + (kk & 3) * 32), id_s, kk ? 1u : 0u);
          if (kk < p.kq)
            umma_tf32(tmem + (uint32_t)(b * 128), desc_k(aQ + kk * 32), desc_k(aKk + kk * 32), id_s, kk ? 1u : 0u);
        }
        umma_commit(&km_empty[s]);
        umma_commit(&sd_full[b]);
      }
      __syncwarp();
    };
    issue_sd(0);
    for (int j = 0; j < nkt; ++j) {
      if (j + 1 < nkt) issue_sd(j + 1);
      const int s = j % p.ns_a, b = j & 1;
      const uint32_t aKm = aR + s * stage_bytes + 8192 + p.vg * 8192;
      bwait(&ds_ready[b], (j >> 1) & 1);
      bwait(&mn_full[s], (j / p.ns_a) & 1);
      fence_after();
      if (lane == 0) {
        for (int kk = 0; kk < AT_TK / 8; ++kk)           // A = dS from TMEM (it replaced S)
          umma_tf32_ts(tmem + 256, tmem + (uint32_t)(b * 128 + kk * 8), desc_mn(aKm + (kk >> 2) * 4096 + (kk & 3) * 1024), id_dq,
                       (j | kk) ? 1u : 0u);
        umma_commit(&dq_done[b]);
        umma_commit(&mn_empty[s]);
        if (j == nkt - 1) umma_commit(dq_full);
      }
      __syncwarp();
    }
  } else {
    const int quarter = warp & 3, half = (warp - 2) >> 2, row = quarter * 32 + lane;
    const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 32);
    const long long grow = (long long)img * p.lq + q0 + row;
    const float lse2 = p.lse[grow] * AT_LOG2E, dsum = p.dsum[grow];
    for (int j = 0; j < nkt; ++j) {
      const int b = j & 1;
      bwait(&sd_full[b], (j >> 1) & 1);
      fence_after();
      uint32_t rs[32], rd[32];
      tmem_ld32(tl + (uint32_t)(b * 128), rs);
      tmem_ld32(tl + (uint32_t)(b * 128 + 64), rd);
      float ds[32];
#pragma unroll
      for (int i = 0; i < 32; ++i)
        ds[i] = rnd_tf32(ex2(fmaf(__uint_as_float(rs[i]), AT_LOG2E, -lse2)) * (__uint_as_float(rd[i]) - dsum));
      tmem_st32(tl + (uint32_t)(b * 128), ds);
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ds_ready[b]);
    }
    bwait(dq_full, 0);
    fence_after();
    if (half == 0) store_acc_row(p.out + grow * p.dk, tmem + ((uint32_t)(quarter * 32) << 16) + 256, p.dk, 1.0f, 0, 1);
    fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// ---------------------------------------------------------------------------------------------------- backward: dK, dV
// One CTA per 128 keys; query tiles of 64.  S^T = K Q^T and dP^T = V dO^T (M = keys, N = queries) so that P^T and dS^T come out
// in the A-operand orientation of dV += P^T dO and dK += dS^T Q — and stay in TMEM, where they replace S^T and dP^T.
// shared memory: K 16 KB | V vg x 16 KB | ring ns_a x [Q (K-major, 64 q) 8 KB | dO (K-major) vg x 8 KB] |
// ring ns_b x [Q (MN-major) 8 KB | dO (MN-major) vg x 8 KB] | lse, D of the query tile 2 x 2 x 64 floats | barriers.
// TMEM (512 columns): buffer b @ b*128: S^T -> P^T @+0, dP^T -> dS^T @+64; dK @256; dV @320.
__global__ void __launch_bounds__(AT_THREADS, 1)
attn_bwd_dkv_kernel(const __grid_constant__ CUtensorMap tm_k, const __grid_constant__ CUtensorMap tm_vk,
                    const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_do,
                    const __grid_constant__ CUtensorMap tm_qm, const __grid_constant__ CUtensorMap tm_dom, const AtParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int stage_bytes = 8192 + p.vg * 8192;
  uint8_t* sK = smem;
  uint8_t* sV = sK + 16384;
  uint8_t* ringk = sV + p.vg * 16384;                        // K-major Q / dO tiles
  uint8_t* ringm = ringk + p.ns_a * stage_bytes;             // MN-major Q / dO tiles
  float* sL = reinterpret_cast<float*>(ringm + p.ns_b * stage_bytes);        // [2][64] lse * log2(e)
  float* sD = sL + 128;                                      // [2][64]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sD + 128);
  uint64_t* kv_full = bars;
  uint64_t* qk_full = bars + 1;                     // AT_MAX_STAGES each
  uint64_t* qk_empty = qk_full + AT_MAX_STAGES;
  uint64_t* qm_full = qk_empty + AT_MAX_STAGES;
  uint64_t* qm_empty = qm_full + AT_MAX_STAGES;
  uint64_t* sd_full = qm_empty + AT_MAX_STAGES;     // 2
  uint64_t* pt_ready = sd_full + 2;                 // 2: P^T and dS^T are back in TMEM
  uint64_t* acc_done = pt_ready + 2;                // 2: dV / dK products of the buffer retired
  uint64_t* acc_full = acc_done + 2;                // 24 barriers
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_full + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k0 = blockIdx.x * AT_TQ, img = blockIdx.y;
  const int nqt = p.lq / AT_TK;

  if (warp == 1) {
    if (lane == 0) {
      mbar_init(kv_full, 1);
      for (int s = 0; s < AT_MAX_STAGES; ++s) {
        mbar_init(&qk_full[s], 1); mbar_init(&qk_empty[s], 1); mbar_init(&qm_full[s], 1); mbar_init(&qm_empty[s], 1);
      }
      for (int s = 0; s < 2; ++s) { mbar_init(&sd_full[s], 1); mbar_init(&pt_ready[s], AT_SWARPS); mbar_init(&acc_done[s], 1); }
      mbar_init(acc_full, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc(tmem_ptr, 512);
  }
  fence_before();
  __syncthreads();
  fence_after();
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    if (lane == 0) {
      mbar_expect_tx(kv_full, (uint32_t)(16384 + p.vg * 16384));
      tma_load_4d(sK, &tm_k, kv_full, 0, k0, 0, img);
      for (int g = 0; g < p.vg; ++g) tma_load_4d(sV + g * 16384, &tm_vk, kv_full, g * 32, k0, 0, img);
      int kt = 0, mt = 0;
      long long t_last = clock64();
      while (kt < nqt || mt < nqt) {
        bool progress = false;
        if (kt < nqt) {
          const int s = kt % p.ns_a;
          if (btest(&qk_empty[s], ((kt / p.ns_a) & 1) ^ 1)) {
            uint8_t* st = ringk + s * stage_bytes;
            mbar_expect_tx(&qk_full[s], (uint32_t)stage_bytes);
            tma_load_4d(st, &tm_q, &qk_full[s], 0, kt * AT_TK, 0, img);
            for (int g = 0; g < p.vg; ++g) tma_load_4d(st + 8192 + g * 8192, &tm_do, &qk_full[s], g * 32, kt * AT_TK, 0, img);
            ++kt; progress = true;
          }
        }
        if (mt < nqt) {
          const int s = mt % p.ns_b;
          if (btest(&qm_empty[s], ((mt / p.ns_b) & 1) ^ 1)) {
            uint8_t* st = ringm + s * stage_bytes;
            mbar_expect_tx(&qm_full[s], (uint32_t)stage_bytes);
            for (int kb = 0; kb < 2; ++kb) {
              tma_load_4d(st + kb * 4096, &tm_qm, &qm_full[s], 0, mt * AT_TK + kb * 32, 0, img);
              for (int g = 0; g < p.vg; ++g)
                tma_load_4d(st + 8192 + (kb * p.vg + g) * 4096, &tm_dom, &qm_full[s], g * 32, mt * AT_TK + kb * 32, 0, img);
            }
            ++mt; progress = true;
          }
        }
        if (progress) t_last = clock64(); else poll_idle(t_last);
      }
    }
  } else if (warp == 1) {
    const uint32_t id_s = idesc(AT_TK, 0), id_dk = idesc(32, 1), id_dv = idesc(p.nv, 1);
    const uint32_t aK = smem_u32(sK), aV = smem_u32(sV), aRk = smem_u32(ringk), aRm = smem_u32(ringm);
    bwait(kv_full, 0);
    auto issue_sd = [&](int i) {
      const int b = i & 1, s = i % p.ns_a;
      const uint32_t aQk = aRk + s * stage_bytes, adOk = aQk + 8192;
      bwait(&qk_full[s], (i / p.ns_a) & 1);
      if (i >= 2) bwait(&acc_done[b], ((i - 2) >> 1) & 1);
      fence_after();
      if (lane == 0) {
        for (int kk = 0; kk < p.kv; ++kk) {              // alternate the two independent accumulations (see the dQ kernel)
          umma_tf32(tmem + (uint32_t)(b * 128 + 64), desc_k(aV + (kk >> 2) * 16384 + (kk & 3) * 32),
                    desc_k(adOk + (kk >> 2) * 8192 + (kk & 3) * 32), id_s, kk ? 1u : 0u);
          if (kk < p.kq)
            umma_tf32(tmem + (uint32_t)(b * 128), desc_k(aK + kk * 32), desc_k(aQk + kk * 32), id_s, kk ? 1u : 0u);
        }
        umma_commit(&qk_empty[s]);
        umma_commit(&sd_full[b]);
      }
      __syncwarp();
    };
    issue_sd(0);
    for (int i = 0; i < nqt; ++i) {
      if (i + 1 < nqt) issue_sd(i + 1);
      const int s = i % p.ns_b, b = i & 1;
      const uint32_t aQm = aRm + s * stage_bytes, adOm = aQm + 8192;
      bwait(&pt_ready[b], (i >> 1) & 1);
      bwait(&qm_full[s], (i / p.ns_b) & 1);
      fence_after();
      if (lane == 0) {
        for (int kk = 0; kk < AT_TK / 8; ++kk) {         // alternately: dV += P^T dO (A = P^T from TMEM), dK += dS^T Q (A = dS^T)
          umma_tf32_ts(tmem + 320, tmem + (uint32_t)(b * 128 + kk * 8), desc_mn(adOm + (kk >> 2) * p.vg * 4096 + (kk & 3) * 1024),
                       id_dv, (i | kk) ? 1u : 0u);
          umma_tf32_ts(tmem + 256, tmem + (uint32_t)(b * 128 + 64 + kk * 8), desc_mn(aQm + (kk >> 2) * 4096 + (kk & 3) * 1024), id_dk,
                       (i | kk) ? 1u : 0u);
        }
        umma_commit(&acc_done[b]);
        umma_commit(&qm_empty[s]);
        if (i == nqt - 1) umma_commit(acc_full);
      }
      __syncwarp();
    }
  } else {
    const int quarter = warp & 3, half = (warp - 2) >> 2, row = quarter * 32 + lane;
    const int st = threadIdx.x - 64;             // 0..255 among the softmax threads
    const uint32_t tl = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(half * 32);
    // per-query lse and D of a tile (columns here) are staged in shared memory and read as broadcasts; the global loads for
    // tile i + 1 are issued at the top of tile i so that their latency is off the per-tile critical path
    const long long gq0 = (long long)img * p.lq + (st < AT_TK ? st : 0);
    float nl = 0.f, nd = 0.f;
    if (st < AT_TK) { nl = p.lse[gq0]; nd = p.dsum[gq0]; }
    for (int i = 0; i < nqt; ++i) {
      const int b = i & 1;
      // buffer b was last read two tiles ago, and every softmax thread has passed the barrier of the tile in between
      if (st < AT_TK) {
        sL[b * AT_TK + st] = nl * AT_LOG2E;
        sD[b * AT_TK + st] = nd;
        if (i + 1 < nqt) { nl = p.lse[gq0 + (i + 1) * AT_TK]; nd = p.dsum[gq0 + (i + 1) * AT_TK]; }
      }
      softmax_bar();
      bwait(&sd_full[b], (i >> 1) & 1);
      fence_after();
      uint32_t rs[32], rd[32];
      tmem_ld32(tl + (uint32_t)(b * 128), rs);
      tmem_ld32(tl + (uint32_t)(b * 128 + 64), rd);
      float pt[32], ds[32];
      const float* lrow = sL + b * AT_TK + half * 32;
      const float* drow = sD + b * AT_TK + half * 32;
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float pe = ex2(fmaf(__uint_as_float(rs[c]), AT_LOG2E, -lrow[c]));
        pt[c] = rnd_tf32(pe);
        ds[c] = rnd_tf32(pe * (__uint_as_float(rd[c]) - drow[c]));
      }
      tmem_st32(tl + (uint32_t)(b * 128), pt);
      tmem_st32(tl + (uint32_t)(b * 128 + 64), ds);
      fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&pt_ready[b]);
    }
    bwait(acc_full, 0);
    fence_after();
    const long long grow = (long long)img * p.lk + k0 + row;
    const uint32_t tq = tmem + ((uint32_t)(quarter * 32) << 16);
    if (half == 1) store_acc_row(p.out + grow * p.dk, tq + 256, p.dk, 1.0f, 0, 1);
    store_acc_row(p.out2 + grow * p.dv, tq + 320, p.dv, 1.0f, half, 2);
    fence_before();
  }
  __syncthreads();
  if (warp == 1) {
    fence_after();
    tmem_dealloc(tmem, 512);
  }
}

__global__ void round_tf32_kernel(float* __restrict__ y, const float* __restrict__ x, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = rna_tf32(x[i]);
}

// [batch, rows, ch] fp32 tensor seen as {ch, rows, 1, batch}; box = 32 channels x box_rows rows
bool make_rows_map(CUtensorMap* tm, const float* base, int ch, int rows, int batch, int box_rows, bool mn_major) {
  return make_act_map(tm, base, ch, rows, 1, batch, ch, (long long)rows * ch, (long long)rows * ch, box_rows, 1, 1,
                      mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B);
}

bool shape_ok(int batch, int lq, int lk, int dk, int dv) {
  return batch >= 1 && batch <= 65535 && lq >= 128 && lq % 128 == 0 && lk >= 128 && lk % 128 == 0 && dk >= 4 && dk <= 32 &&
         dk % 4 == 0 && dv >= 16 && dv <= 128 && dv % 16 == 0;      // (dv = 128: one stage per ring in the dK/dV kernel still fits)
}

void fill_params(AtParams* p, int lq, int lk, int dk, int dv) {
  memset(p, 0, sizeof(*p));
  p->lq = lq; p->lk = lk; p->dk = dk; p->dv = dv;
  p->kq = (dk + 7) / 8; p->kv = (dv + 7) / 8; p->vg = (dv + 31) / 32; p->nv = dv;
}

template <typename F>
int set_smem(cgan_ctx* ctx, F* kernel, size_t bytes, const char* who) {
  if (bytes > 227 * 1024) return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: shared memory%s", who);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: %s", who, cudaGetErrorString(e));
  return CGAN_OK;
}

}  // namespace

extern "C" {

int cgan_round_tf32(cgan_ctx* ctx, float* y, const float* x, int64_t n) {
  if (!ctx) return CGAN_ERR_ARG;
  CGAN_REQUIRE(ctx, y && x && n >= 0, "bad argument");
  if (n == 0) return CGAN_OK;
  long long blocks = (n + 255) / 256, cap = (long long)ctx->num_sms * 16;
  round_tf32_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, ctx->stream>>>(y, x, n);
  CGAN_LAUNCHED(ctx);
  return CGAN_OK;
}

int cgan_attention_supported(cgan_ctx* ctx, int batch, int lq, int lk, int dk, int dv) {
  return (ctx && ctx->math_mode == 1 && shape_ok(batch, lq, lk, dk, dv) && get_encode()) ? 1 : 0;
}

int cgan_attention_fwd(cgan_ctx* ctx, const float* q, const float* k, const float* v, float* out, float* lse, int batch, int lq,
                       int lk, int dk, int dv) {
  if (!ctx) return CGAN_ERR_ARG;
  CGAN_REQUIRE(ctx, q && k && v && out && lse, "null pointer");
  if (!cgan_attention_supported(ctx, batch, lq, lk, dk, dv))
    return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: needs math_mode 1, lq, lk multiples of 128, dk <= 32 (x4), dv <= 128 (x16)%s",
                     "cgan_attention_fwd");
  AtParams p;
  fill_params(&p, lq, lk, dk, dv);
  p.out = out; p.out2 = lse;
  CUtensorMap tq, tk, tv;
  if (!make_rows_map(&tq, q, dk, lq, batch, 128, false) || !make_rows_map(&tk, k, dk, lk, batch, 64, false) ||
      !make_rows_map(&tv, v, dv, lk, batch, 32, true))
    return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed%s", "cgan_attention_fwd");
  // Two CTAs per SM (256 TMEM columns each) with rings as deep as half an SM's shared memory allows.  Measured
  // (profiles/r2_attention_*.txt): two resident CTAs overlap each other's per-tile dependency chains better than deeper
  // prefetch in one CTA per SM (1.18 ms against 2.04 ms).
  const size_t v_stage = (size_t)p.vg * 8192, fixed = 16384 + 1280 + 1024;
  const size_t budget = (AT_SMEM_MAX - 2048) / 2;
  p.ns_a = AT_MAX_STAGES;
  p.ns_b = (int)((budget - fixed - (size_t)p.ns_a * 8192) / v_stage);
  if (p.ns_b > AT_MAX_STAGES) p.ns_b = AT_MAX_STAGES;
  if (p.ns_b > lk / AT_TK) p.ns_b = lk / AT_TK;
  if (p.ns_b < 1) return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: shared memory%s", "cgan_attention_fwd");
  const size_t smem = fixed + (size_t)p.ns_a * 8192 + (size_t)p.ns_b * v_stage;
  int rc = set_smem(ctx, attn_fwd_kernel, smem, "cgan_attention_fwd");
  if (rc) return rc;
  attn_fwd_kernel<<<dim3(lq / AT_TQ, batch), AT_THREADS, smem, ctx->stream>>>(tq, tk, tv, p);
  CGAN_LAUNCHED(ctx);
  ctx->last_path = CGAN_PATH_TCGEN05_TF32;
  return CGAN_OK;
}

int cgan_attention_bwd(cgan_ctx* ctx, const float* q, const float* k, const float* v, const float* out, const float* lse,
                       const float* dout, float* dq, float* dk_out, float* dv_out, int batch, int lq, int lk, int dk, int dv) {
  if (!ctx) return CGAN_ERR_ARG;
  CGAN_REQUIRE(ctx, q && k && v && out && lse && dout && dq && dk_out && dv_out, "null pointer");
  if (!cgan_attention_supported(ctx, batch, lq, lk, dk, dv))
    return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: unsupported shape or math mode%s", "cgan_attention_bwd");
  void* ws = nullptr;
  int rc = cgan_ws(ctx, (size_t)batch * lq * sizeof(float), &ws);
  if (rc) return rc;
  float* dsum = reinterpret_cast<float*>(ws);
  rc = cgan_rowdot(ctx, dsum, dout, out, (int64_t)batch * lq, dv);          // D = rowsum(dO * O)
  if (rc) return rc;
  AtParams p;
  fill_params(&p, lq, lk, dk, dv);
  p.lse = lse; p.dsum = dsum;
  CUtensorMap tq128, tdo128, tk64, tvk64, tkm, tk128, tvk128, tq64, tdo64, tqm, tdom;
  if (!make_rows_map(&tq128, q, dk, lq, batch, 128, false) || !make_rows_map(&tdo128, dout, dv, lq, batch, 128, false) ||
      !make_rows_map(&tk64, k, dk, lk, batch, 64, false) || !make_rows_map(&tvk64, v, dv, lk, batch, 64, false) ||
      !make_rows_map(&tkm, k, dk, lk, batch, 32, true) || !make_rows_map(&tk128, k, dk, lk, batch, 128, false) ||
      !make_rows_map(&tvk128, v, dv, lk, batch, 128, false) || !make_rows_map(&tq64, q, dk, lq, batch, 64, false) ||
      !make_rows_map(&tdo64, dout, dv, lq, batch, 64, false) || !make_rows_map(&tqm, q, dk, lq, batch, 32, true) ||
      !make_rows_map(&tdom, dout, dv, lq, batch, 32, true))
    return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed%s", "cgan_attention_bwd");
  {
    p.out = dq; p.out2 = nullptr;
    const size_t fixed = 16384 + (size_t)p.vg * 16384 + 256 + 1024, stage = 16384 + (size_t)p.vg * 8192;
    p.ns_a = (int)((AT_SMEM_MAX - fixed) / stage);
    if (p.ns_a > AT_MAX_STAGES) p.ns_a = AT_MAX_STAGES;
    if (p.ns_a > lk / AT_TK) p.ns_a = lk / AT_TK;
    p.ns_b = p.ns_a;
    const size_t smem = fixed + (size_t)p.ns_a * stage;
    rc = set_smem(ctx, attn_bwd_dq_kernel, smem, "cgan_attention_bwd");
    if (rc) return rc;
    attn_bwd_dq_kernel<<<dim3(lq / AT_TQ, batch), AT_THREADS, smem, ctx->stream>>>(tq128, tdo128, tk64, tvk64, tkm, p);
    CGAN_LAUNCHED(ctx);
  }
  {
    p.out = dk_out; p.out2 = dv_out;
    const size_t fixed = 16384 + (size_t)p.vg * 16384 + 1024 + 256 + 1024, stage = 8192 + (size_t)p.vg * 8192;
    int total = (int)((AT_SMEM_MAX - fixed) / stage);
    if (total > 2 * AT_MAX_STAGES) total = 2 * AT_MAX_STAGES;
    p.ns_a = (total + 1) / 2;           // K-major group: needed first (S^T, dP^T)
    p.ns_b = total / 2;                 // MN-major group (dV, dK)
    if (p.ns_a > lq / AT_TK) p.ns_a = lq / AT_TK;
    if (p.ns_b > lq / AT_TK) p.ns_b = lq / AT_TK;
    const size_t smem = fixed + (size_t)(p.ns_a + p.ns_b) * stage;
    rc = set_smem(ctx, attn_bwd_dkv_kernel, smem, "cgan_attention_bwd");
    if (rc) return rc;
    attn_bwd_dkv_kernel<<<dim3(lk / AT_TQ, batch), AT_THREADS, smem, ctx->stream>>>(tk128, tvk128, tq64, tdo64, tqm, tdom, p);
    CGAN_LAUNCHED(ctx);
  }
  ctx->last_path = CGAN_PATH_TCGEN05_TF32;
  return CGAN_OK;
}

}  // extern "C"
