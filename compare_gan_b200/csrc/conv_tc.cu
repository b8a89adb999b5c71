// tcgen05 (5th-gen tensor core) implicit-GEMM convolution for sm_100a — math_mode 1.
//
//   out[pixel, co] = sum_{tap, ci} in[pixel + off(tap), ci] * wt[tap][co][ci]        (+ bias[co])
//
// * A operand (activations, NHWC fp32): one TMA 4-D tiled load per (tap, 32-channel chunk) brings a
//   [images x rows x cols x 32ch] box = 128 pixels x 128 B straight into the 128B-swizzled K-major layout
//   the UMMA descriptor expects; TF SAME padding is the TMA out-of-bounds zero fill (negative coordinates),
//   so no im2col buffer and no padding pass exist.
// * B operand (weights): pre-rounded (round-to-nearest TF32) and laid out [tap][row][k] K-major by a small
//   prep kernel; TMA 3-D loads.
// * The fp32 activations are rounded to nearest TF32 IN SHARED MEMORY by the (otherwise idle) epilogue
//   warps before the tensor core reads them — tcgen05 kind::tf32 would otherwise truncate the low 13 bits,
//   a systematic -2^-11 relative bias per product that accumulates through a 13-layer discriminator.
// * D accumulates in TMEM (128 lanes x N fp32 columns); one elected thread issues tcgen05.mma
//   (M=128, N<=256, K=8 per instruction); completion is tracked with tcgen05.commit -> mbarrier.
// * Warp roles: warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer, warps 2..5 = operand
//   rounding during the main loop, then epilogue (tcgen05.ld -> +bias -> global).
//
// The same kernel serves forward and input-gradient convolutions (and the four sub-pixel phases of a
// conv over a zero-inserted 2x upsampled input): the host supplies, per tap, the input offset and the weight
// slice, and the output pixel strides.
#include "tc_common.cuh"

namespace {

using namespace tc;

constexpr int TC_BM = 128;          // output pixels per CTA tile (UMMA M)
constexpr int TC_BK = 32;           // fp32 channels per k-block: 128 B = one swizzle row
constexpr int TC_MAX_STAGES = 4;   // the pipeline depth is chosen per launch so that TWO CTAs fit an SM (see host code)
constexpr int TC_MAX_TAPS = 32;
constexpr int TC_RWARPS = 8;         // warps 2..9: operand rounding, then the epilogue (two warps per TMEM lane quarter)
constexpr int TC_THREADS = 64 + 32 * TC_RWARPS;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 4;     // 16 KB

struct TcParams {
  int ntaps, kchunks;               // k-blocks = ntaps * kchunks
  int off_h[TC_MAX_TAPS], off_w[TC_MAX_TAPS], wtap[TC_MAX_TAPS], amap[TC_MAX_TAPS];   // amap: which input view
  int bw, bh, bni;                  // tile box: bw*bh*bni == 128
  int tiles_w, tiles_h;             // tiles per image row / column
  int rows_used;                    // bw*bh*bni <= 128 pixel rows actually filled by the TMA box
  int img_n, img_h, img_w;          // extent of the pixel grid (tiles at the border hang over; those rows are not stored)
  int relu;                         // fused ReLU in the epilogue
  int round_a;                      // 1: round the activation tiles to nearest TF32 in shared memory (operand not pre-rounded)
  int round_out;                    // 1: store TF32-rounded outputs (the consumer is another tensor-core contraction)
  float mask_leak;                  // with `mask`: out = ref > 0 ? v : mask_leak * v  ((leaky-)ReLU backward fused into a dgrad)
  const float* residual;            // optional tensor of the output's geometry added before the activation (residual blocks)
  const float* mask;                // optional tensor of the output's geometry: the (leaky-)ReLU input/output whose sign gates v
  int wimg_stride;                  // batched GEMM: weight slice = wtap + image * wimg_stride (tiles never span images)
  int bn;                           // UMMA N (multiple of 32, <= 256)
  int stages;                       // smem pipeline depth (2..4)
  int mt;                           // pixel tiles per CTA sharing one weight tile (accumulators mt x bn TMEM columns)
  int tiles_total;                  // tiles_w * tiles_h * tiles_n
  int tmem_cols;                    // power of two >= bn
  int cout;                         // valid output channels (row length of `out` pixels)
  long long s_n, s_h, s_w, base;    // output element strides / offset (floats)
  float* out;
  const float* bias;
  // halo mode (conv_tc_halo_kernel): the taps come in `hg` groups of `hnv` vertically consecutive taps that share their
  // horizontal offset; one TMA box of bh + hnv - 1 rows serves all taps of a group (the vertical shift is a descriptor
  // offset of bw rows), so the activation operand crosses L2 -> smem `hg` times per channel chunk instead of hg * hnv
  // sub-pixel phases merged into one launch (blockIdx.z): phase ph owns the taps [ph_tap0[ph], ph_tap0[ph+1]) and writes
  // at element offset ph_base[ph] (a convolution over a zero-inserted input, a stride-2 input gradient)
  int nphases;
  int ph_tap0[5];
  long long ph_base[4];
  int hg, hnv;
  int h_off_w[4], h_off_h0[4], h_wtap[4][4];
  int a_halo_bytes;                 // smem footprint of one tile's halo box (1024-aligned)
  int a_box_bytes;                  // bytes TMA writes per halo box
  int sa_stages, sb_stages;
};

// K-major, 128B-swizzled shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm100):
// start>>4 [0,14) | LBO>>4 [16,30) (unused for swizzled K-major, 1) | SBO>>4 [32,46) = 1024 B between 8-row groups
// | version=1 [46,48) | layout SWIZZLE_128B=2 [61,64)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}

// up to four views of the input tensor (the sub-pixel phases of a 2x-upsampled gradient); plain convs use view 0
struct AMaps { CUtensorMap m[4]; };


__device__ __forceinline__ void tc_tile_origin(const TcParams& p, int t, int& ow0, int& oh0, int& n0) {
  const int tw = t % p.tiles_w; t /= p.tiles_w;
  const int th = t % p.tiles_h;
  const int tn = t / p.tiles_h;
  ow0 = tw * p.bw; oh0 = th * p.bh; n0 = tn * p.bni;
}

// Epilogue of warps 2..9: tcgen05.ld the accumulators of this CTA's tiles, apply bias / residual / ReLU / mask / TF32
// rounding, store.  TMEM lane quarter is fixed by (warp id % 4); row of the tile = TMEM lane.
//
// tcgen05.ld hands every thread 32 consecutive columns of ITS row; storing them from there costs one 16-byte piece in
// each of 32 different 128-byte lines per instruction — 32 LSU wavefronts, and the epilogue (a fifth of the kernel at
// one CTA per SM, ncu r2: 129 k wavefronts per SM) is bound by exactly that.  Each warp therefore transposes its
// 32 x 32 chunk through a private 32 x 36-float staging area in the (by now idle) operand ring, after which a quarter
// warp owns one row's 128 contiguous bytes: 4 wavefronts per store instruction, and the fused residual / mask reads
// coalesce the same way.  `stg` = shared address of this warp's staging area.
constexpr int TC_STG_ROW_BYTES = 36 * 4;                     // 32 columns + 16 B pad: 16-byte aligned, conflict-free v4 access
constexpr int TC_STG_WARP_BYTES = 32 * TC_STG_ROW_BYTES;     // 4608 B per warp, 36 KB per CTA (every operand ring holds >= 40 KB)

__device__ __forceinline__ float4 tc_out_math(const TcParams& p, float4 v, const float4 bv, long long off) {
  v.x += bv.x; v.y += bv.y; v.z += bv.z; v.w += bv.w;
  if (p.residual) {
    const float4 rv = *reinterpret_cast<const float4*>(p.residual + off);
    v.x += rv.x; v.y += rv.y; v.z += rv.z; v.w += rv.w;
  }
  if (p.relu) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
  if (p.mask) {
    const float4 mv = *reinterpret_cast<const float4*>(p.mask + off);
    v.x = mv.x > 0.f ? v.x : p.mask_leak * v.x; v.y = mv.y > 0.f ? v.y : p.mask_leak * v.y;
    v.z = mv.z > 0.f ? v.z : p.mask_leak * v.z; v.w = mv.w > 0.f ? v.w : p.mask_leak * v.w;
  }
  if (p.round_out) { v.x = rna_tf32(v.x); v.y = rna_tf32(v.y); v.z = rna_tf32(v.z); v.w = rna_tf32(v.w); }
  return v;
}

__device__ __forceinline__ void tc_store_tiles(const TcParams& p, uint32_t tmem_base, int tile0, int nt_here, int nb0,
                                               int warp, int lane, long long out_base, uint32_t stg) {
  const int quarter = warp & 3;
  const int m = quarter * 32 + lane;
  const int wi = m % p.bw;
  const int hi = (m / p.bw) % p.bh;
  const int ni = m / (p.bw * p.bh);
  const int sub = lane >> 3, c4 = (lane & 7) * 4;       // transposed role: row (i*4 + sub) of the chunk, columns c4..c4+3
  asm volatile("" : "+r"(stg));      // held in a register: ptxas would otherwise recompute it after every tcgen05.ld
  for (int tl = 0; tl < nt_here; ++tl) {
    int ow0, oh0, n0;
    tc_tile_origin(p, tile0 + tl, ow0, oh0, n0);
    // rows beyond the box (stale smem) and pixels outside the grid are computed but never stored
    const bool row_ok = m < p.rows_used && n0 + ni < p.img_n && oh0 + hi < p.img_h && ow0 + wi < p.img_w;
    // element offset of this row's first column in `out` (residual / mask share the output's geometry)
    const long long roff = out_base + (long long)(n0 + ni) * p.s_n + (long long)(oh0 + hi) * p.s_h +
                           (long long)(ow0 + wi) * p.s_w + nb0;
    const uint32_t okmask = __ballot_sync(0xffffffffu, row_ok);
    long long roffs[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) roffs[i] = __shfl_sync(0xffffffffu, roff, i * 4 + sub);
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(tl * p.bn);
    // two warps share a lane quarter: the first takes the lower half of the 32-column chunks, the second the rest
    const int nchunks = p.bn / 32, csplit = (nchunks + 1) / 2;
    const int cbeg = (warp - 2) < 4 ? 0 : csplit * 32, cend = (warp - 2) < 4 ? csplit * 32 : p.bn;
    for (int c0 = cbeg; c0 < cend; c0 += 32) {
      uint32_t r[32];
      tmem_ld32(taddr + (uint32_t)c0, r);
      const bool whole = nb0 + c0 + 32 <= p.cout && (p.cout & 3) == 0;      // warp-uniform
      if (whole) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          sts128(stg + lane * TC_STG_ROW_BYTES + j * 16,
                 make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                             __uint_as_float(r[4 * j + 3])));
        __syncwarp();
        float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) bv = *reinterpret_cast<const float4*>(p.bias + nb0 + c0 + c4);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 v = lds128(stg + (i * 4 + sub) * TC_STG_ROW_BYTES + c4 * 4);
          if ((okmask >> (i * 4 + sub)) & 1u) {
            const long long off = roffs[i] + c0 + c4;
            *reinterpret_cast<float4*>(p.out + off) = tc_out_math(p, v, bv, off);
          }
        }
        __syncwarp();
      } else if (row_ok) {      // thin / padded tile (e.g. the 256->3 image conv): only the first `cout` columns exist
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if (nb0 + c0 + j < p.cout) {
            float v = __uint_as_float(r[j]);
            if (p.bias) v += p.bias[nb0 + c0 + j];
            if (p.residual) v += p.residual[roff + c0 + j];
            if (p.relu) v = fmaxf(v, 0.f);
            if (p.mask) v = p.mask[roff + c0 + j] > 0.f ? v : p.mask_leak * v;
            if (p.round_out) v = rna_tf32(v);
            p.out[roff + c0 + j] = v;
          }
        }
      }
    }
  }
}

__global__ void __launch_bounds__(TC_THREADS, 2)
conv_tc_kernel(const __grid_constant__ AMaps tm_as, const __grid_constant__ CUtensorMap tm_b, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve: [stages][mt x A 16KB][B bn*128B] | barriers | tmem ptr
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_bytes = p.bn * TC_BK * 4;
  const int a_bytes = p.mt * TC_A_BYTES;
  const int stage_bytes = a_bytes + b_bytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + p.stages * stage_bytes);
  uint64_t* ready_bar = full_bar + p.stages;
  uint64_t* empty_bar = ready_bar + p.stages;
  uint64_t* tmem_full_bar = empty_bar + p.stages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tap0 = p.ph_tap0[blockIdx.z];
  const int num_kb = (p.ph_tap0[blockIdx.z + 1] - tap0) * p.kchunks;

  // this CTA's pixel tiles: [tile0, tile0 + nt_here).  They all multiply the same weight tile, which is therefore
  // fetched from L2 once per k-block for mt*128 pixels: the kernel is bound by L2->SM bytes per MMA, not by HBM.
  const int tile0 = blockIdx.x * p.mt;
  const int nt_here = min(p.mt, p.tiles_total - tile0);
  auto tile_origin = [&](int i, int& ow0, int& oh0, int& n0) { tc_tile_origin(p, tile0 + i, ow0, oh0, n0); };
  const int nb0 = blockIdx.y * p.bn;          // first output channel of this CTA

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_as.m[0]) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_b) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < p.stages; ++s) {
        mbar_init(&full_bar[s], 1);
        mbar_init(&ready_bar[s], TC_RWARPS);      // one arrive per rounding warp
        mbar_init(&empty_bar[s], 1);
      }
      mbar_init(tmem_full_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    // TMEM: 256 fp32 columns x 128 lanes for the accumulator
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        const int tl = kb / p.kchunks, kc = kb - tl * p.kchunks, tap = tap0 + tl;
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * stage_bytes;
        uint8_t* sb = sa + a_bytes;
        mbar_expect_tx(&full_bar[stage], (uint32_t)(nt_here * p.rows_used * TC_BK * 4 + b_bytes));
        int ow0, oh0, n0;
        for (int i = 0; i < nt_here; ++i) {
          tile_origin(i, ow0, oh0, n0);
          tma_load_4d(sa + i * TC_A_BYTES, &tm_as.m[p.amap[tap]], &full_bar[stage], kc * TC_BK, ow0 + p.off_w[tap],
                      oh0 + p.off_h[tap], n0);
        }
        tile_origin(0, ow0, oh0, n0);           // batched GEMM: all tiles of a CTA lie in one image (host guarantees)
        tma_load_3d(sb, &tm_b, &full_bar[stage], kc * TC_BK, nb0, p.wtap[tap] + n0 * p.wimg_stride);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    // instruction descriptor (cute::UMMA::InstrDescriptor): D=F32 (1<<4), A=TF32 (2<<7), B=TF32 (2<<10), K-major A/B,
    // N>>3 at [17,23), M>>4 at [24,29)
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(p.round_a ? &ready_bar[stage] : &full_bar[stage], phase);   // pre-rounded operands: straight from TMA
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (lane == 0) {
        const uint32_t a_addr = smem_u32(smem + stage * stage_bytes);
        const uint32_t b_addr = a_addr + a_bytes;
        for (int i = 0; i < nt_here; ++i) {
#pragma unroll
          for (int k = 0; k < TC_BK / 8; ++k) {     // UMMA_K = 8 for tf32: 32 B per step inside the 128 B swizzle row
            umma_tf32(tmem_base + (uint32_t)(i * p.bn), make_desc(a_addr + i * TC_A_BYTES + k * 32), make_desc(b_addr + k * 32),
                      idesc, (kb | k) ? 1u : 0u);
          }
        }
        umma_commit(&empty_bar[stage]);              // frees the smem slot when these MMAs retire
        if (kb == num_kb - 1) umma_commit(tmem_full_bar);
      }
      __syncwarp();
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
  } else {
    // ===== warps 2..9: round A to nearest TF32 in smem, then epilogue =====
    const int q = threadIdx.x - 64;                  // 0..255
    if (p.round_a) {
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        uint32_t a4 = smem_u32(smem + stage * stage_bytes) + q * 16;
        for (int tl = 0; tl < nt_here; ++tl, a4 += TC_A_BYTES) {
          float4 v[TC_A_BYTES / 16 / (32 * TC_RWARPS)];       // 1024 float4 / 256 threads = 4 each, loads first
#pragma unroll
          for (int i = 0; i < TC_A_BYTES / 16 / (32 * TC_RWARPS); ++i) v[i] = lds128(a4 + i * (512 * TC_RWARPS));
#pragma unroll
          for (int i = 0; i < TC_A_BYTES / 16 / (32 * TC_RWARPS); ++i) {
            v[i].x = rna_tf32(v[i].x); v[i].y = rna_tf32(v[i].y); v[i].z = rna_tf32(v[i].z); v[i].w = rna_tf32(v[i].w);
            sts128(a4 + i * (512 * TC_RWARPS), v[i]);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async proxy (UMMA) reads
        __syncwarp();
        if (lane == 0) mbar_arrive(&ready_bar[stage]);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
    mbar_wait(tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tc_store_tiles(p, tmem_base, tile0, nt_here, nb0, warp, lane, p.ph_base[blockIdx.z],
                   smem_u32(smem) + (warp - 2) * TC_STG_WARP_BYTES);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// ---- halo variant ------------------------------------------------------------------------------------------------
// 3x3 stride-1 convolutions (forward and input gradient) are bound by the L2 -> shared-memory operand feed, not by the
// tensor pipe (DESIGN.md section 3): per 32-channel k-block a CTA pulls 16 KB of activations per pixel tile for every one
// of the nine taps although the nine boxes overlap almost completely.  Here the three taps of one kernel COLUMN share a
// single TMA box of bh + 2 image rows; the vertical shift of a tap is a descriptor start-address offset of bw pixel rows
// (a multiple of 1024 B, so the 128B-swizzle phase is unchanged).  The activation operand is fetched 3 x (bh+2)/bh times
// per chunk instead of 9 x (x1.5 instead of x9 at 4-row tiles), which also halves the in-smem rounding work of operands
// that are not pre-rounded.  Activations and weights run in two rings of their own (a halo box lives for three k-blocks).
// Up to four pixel tiles per CTA share each weight tile (mt x bn <= 512 TMEM columns), one CTA per SM.
__global__ void __launch_bounds__(TC_THREADS, 1)
conv_tc_halo_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int b_bytes = p.bn * TC_BK * 4;
  const int a_stage = p.mt * p.a_halo_bytes;
  uint8_t* smem_b = smem + p.sa_stages * a_stage;
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem_b + p.sb_stages * b_bytes);
  uint64_t* a_ready = a_full + p.sa_stages;
  uint64_t* a_empty = a_ready + p.sa_stages;
  uint64_t* b_full = a_empty + p.sa_stages;
  uint64_t* b_empty = b_full + p.sb_stages;
  uint64_t* tmem_full_bar = b_empty + p.sb_stages;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile0 = blockIdx.x * p.mt;
  const int nt_here = min(p.mt, p.tiles_total - tile0);
  const int nb0 = blockIdx.y * p.bn;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tm_b) : "memory");
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < p.sa_stages; ++s) {
        mbar_init(&a_full[s], 1);
        mbar_init(&a_ready[s], TC_RWARPS);
        mbar_init(&a_empty[s], 1);
      }
      for (int s = 0; s < p.sb_stages; ++s) {
        mbar_init(&b_full[s], 1);
        mbar_init(&b_empty[s], 1);
      }
      mbar_init(tmem_full_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"((uint32_t)p.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===== TMA producer: per (channel chunk, tap column) one halo box per tile, then the hnv weight tiles =====
    if (lane == 0) {
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;
      for (int kc = 0; kc < p.kchunks; ++kc) {
        for (int g = 0; g < p.hg; ++g) {
          mbar_wait(&a_empty[sa], pa ^ 1);
          mbar_expect_tx(&a_full[sa], (uint32_t)(nt_here * p.a_box_bytes));
          for (int i = 0; i < nt_here; ++i) {
            int ow0, oh0, n0;
            tc_tile_origin(p, tile0 + i, ow0, oh0, n0);
            tma_load_4d(smem + sa * a_stage + i * p.a_halo_bytes, &tm_a, &a_full[sa], kc * TC_BK, ow0 + p.h_off_w[g],
                        oh0 + p.h_off_h0[g], n0);
          }
          if (++sa == p.sa_stages) { sa = 0; pa ^= 1; }
          for (int t = 0; t < p.hnv; ++t) {
            mbar_wait(&b_empty[sb], pb ^ 1);
            mbar_expect_tx(&b_full[sb], (uint32_t)b_bytes);
            tma_load_3d(smem_b + sb * b_bytes, &tm_b, &b_full[sb], kc * TC_BK, nb0, p.h_wtap[g][t]);
            if (++sb == p.sb_stages) { sb = 0; pb ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.bn >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
    int sa = 0, sb = 0;
    uint32_t pa = 0, pb = 0;
    const uint32_t tap_shift = (uint32_t)(p.bw * 128);          // one image row of the box = bw pixel rows of 128 B
    for (int kc = 0; kc < p.kchunks; ++kc) {
      for (int g = 0; g < p.hg; ++g) {
        mbar_wait(p.round_a ? &a_ready[sa] : &a_full[sa], pa);
        const uint32_t a_addr = smem_u32(smem + sa * a_stage);
        for (int t = 0; t < p.hnv; ++t) {
          mbar_wait(&b_full[sb], pb);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          if (lane == 0) {
            const uint32_t b_addr = smem_u32(smem_b + sb * b_bytes);
            const uint32_t first = (kc | g | t) ? 1u : 0u;
            for (int i = 0; i < nt_here; ++i) {
#pragma unroll
              for (int k = 0; k < TC_BK / 8; ++k)
                umma_tf32(tmem_base + (uint32_t)(i * p.bn), make_desc(a_addr + i * p.a_halo_bytes + t * tap_shift + k * 32),
                          make_desc(b_addr + k * 32), idesc, (first | (uint32_t)k) ? 1u : 0u);
            }
            umma_commit(&b_empty[sb]);
            if (t == p.hnv - 1) umma_commit(&a_empty[sa]);
            if (kc == p.kchunks - 1 && g == p.hg - 1 && t == p.hnv - 1) umma_commit(tmem_full_bar);
          }
          __syncwarp();
          if (++sb == p.sb_stages) { sb = 0; pb ^= 1; }
        }
        if (++sa == p.sa_stages) { sa = 0; pa ^= 1; }
      }
    }
  } else {
    // ===== warps 2..9: round the halo boxes to nearest TF32 in smem (operand not pre-rounded), then the epilogue =====
    if (p.round_a) {
      const int q = threadIdx.x - 64;
      const int n16 = p.a_box_bytes / 16;            // float4s per box (a multiple of 32 * TC_RWARPS, host-checked)
      int sa = 0;
      uint32_t pa = 0;
      for (int it = 0; it < p.kchunks * p.hg; ++it) {
        mbar_wait(&a_full[sa], pa);
        for (int tl = 0; tl < nt_here; ++tl) {
          const uint32_t a4 = smem_u32(smem + sa * a_stage + tl * p.a_halo_bytes);
#pragma unroll 2
          for (int i = q; i < n16; i += 32 * TC_RWARPS) {
            float4 v = lds128(a4 + i * 16);
            v.x = rna_tf32(v.x); v.y = rna_tf32(v.y); v.z = rna_tf32(v.z); v.w = rna_tf32(v.w);
            sts128(a4 + i * 16, v);
          }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&a_ready[sa]);
        if (++sa == p.sa_stages) { sa = 0; pa ^= 1; }
      }
    }
    mbar_wait(tmem_full_bar, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    tc_store_tiles(p, tmem_base, tile0, nt_here, nb0, warp, lane, p.base, smem_u32(smem) + (warp - 2) * TC_STG_WARP_BYTES);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  }
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)p.tmem_cols) : "memory");
  }
}

// dst[tap][r][k] (r < rows_pad) = rna_tf32(src[tap][k][r]) (transpose) or rna_tf32(src[tap][r][k]); rows >= `rows` are 0
__global__ void wprep_kernel(float* __restrict__ dst, const float* __restrict__ src, int taps, int rows, int rows_pad,
                             int kdim, int kdim_pad, int transpose) {
  long long tot = (long long)taps * rows_pad * kdim_pad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    int k = (int)(i % kdim_pad);
    long long t = i / kdim_pad;
    int r = (int)(t % rows_pad);
    int tap = (int)(t / rows_pad);
    float v = 0.f;
    if (r < rows && k < kdim)
      v = transpose ? src[((long long)tap * kdim + k) * rows + r] : src[((long long)tap * rows + r) * kdim + k];
    dst[i] = rna_tf32(v);
  }
}

// 128-pixel tile = bni images x bh rows x bw columns (bw*bh*bni <= 128).  Any grid size is accepted: border tiles hang
// over (TMA zero-fills, the epilogue masks), e.g. Inception's 35x35 maps use 35x3 boxes (105 of 128 MMA rows).
inline void tc_geometry(int n, int h, int w, int* bw, int* bh, int* bni, int* tw, int* th, int* tn) {
  int parts = (w + 127) / 128;
  *bw = (w + parts - 1) / parts;
  *tw = (w + *bw - 1) / *bw;
  *bh = 128 / *bw; if (*bh > h) *bh = h; if (*bh < 1) *bh = 1;
  *th = (h + *bh - 1) / *bh;
  *bni = (*bh == h) ? 128 / (*bw * *bh) : 1;
  if (*bni < 1) *bni = 1;
  if (*bni > n) *bni = n;
  *tn = (n + *bni - 1) / *bni;
}

inline int tc_pick_bn(int ncols_pad) {     // largest UMMA N <= 256 (multiple of 32) that divides the padded column count
  if (ncols_pad <= 256) return ncols_pad;
  for (int b = 256; b >= 32; b -= 32)
    if (ncols_pad % b == 0) return b;
  return 0;
}

// Few pixel tiles (8x8 / 17x17 Inception stages at batch 64, the 4x4 GAN stages): the widest column tile would leave SMs
// idle, so the columns are split further (>= 64) until there is at least one CTA per SM.  The K order is unchanged, so
// the result is bit-identical to the wide tile's.
inline int tc_pick_bn_occupancy(int ncols_pad, long long tiles_m, int sms) {
  int best = tc_pick_bn(ncols_pad);
  if (best == 0 || tiles_m * (ncols_pad / best) >= sms) return best;
  int pick = best;
  for (int b = best - 32; b >= 64; b -= 32) {
    if (ncols_pad % b) continue;
    pick = b;
    if (tiles_m * (ncols_pad / b) >= sms) break;
  }
  return pick;
}

}  // namespace

// Geometry the tensor-core path accepts for a stride-1 convolution-like contraction.
bool cgan_tc_shape_ok(int n, int h, int w, int kdim, int ncols) {
  if (n < 1 || h < 1 || w < 1 || ncols < 1) return false;
  if (kdim < 8 || kdim % 4 != 0) return false;           // TMA needs 16-byte pixel strides; K is zero-padded to 32
  if (ncols > 256 && ncols % 32 != 0) return false;      // small column counts are zero-padded to a multiple of 32
  int bn = tc_pick_bn((ncols + 31) / 32 * 32);
  return bn != 0 && bn % 32 == 0;
}

// Weights -> TF32-rounded (nearest) K-major [taps_total][ncols_pad][kdim_pad] in the context workspace.  Split from the
// launch so that a convolution over a zero-inserted input prepares its weights ONCE for its four sub-pixel phases.
int cgan_tc_prep_weights(cgan_ctx* ctx, const float* wsrc, int taps_total, int transpose_w, int ncols, int kdim, float** out) {
  const int kdim_pad = (kdim + TC_BK - 1) / TC_BK * TC_BK;
  const int ncols_pad = (ncols + 31) / 32 * 32;
  void* ws = nullptr;
  size_t wbytes = (size_t)taps_total * ncols_pad * kdim_pad * sizeof(float);
  int rc = cgan_ws(ctx, wbytes, &ws);
  if (rc) return rc;
  float* wt = reinterpret_cast<float*>(ws);
  long long tot = (long long)taps_total * ncols_pad * kdim_pad;
  long long blocks = (tot + 255) / 256, cap = (long long)ctx->num_sms * 8;
  wprep_kernel<<<(int)(blocks > cap ? cap : blocks), 256, 0, ctx->stream>>>(wt, wsrc, taps_total, ncols, ncols_pad, kdim,
                                                                             kdim_pad, transpose_w);
  CGAN_LAUNCHED(ctx);
  *out = wt;
  return CGAN_OK;
}

// in: fp32 NHWC activations seen through `nviews` views of logical size [n, h, w, kdim] (view v starts at
// in + view_off[v], pixel strides sw/sh/sn floats) — one view for ordinary convs, the four sub-pixel phases of a
// 2x-upsampled gradient for the input gradient of a conv over a zero-inserted input.
// wsrc: weights [taps_total][kdim][ncols] (transpose_w=1) or [taps_total][ncols][kdim] (transpose_w=0); ignored when
// ex->wprep holds the output of cgan_tc_prep_weights for the same weights.
// taps: `ntaps` entries (off_h, off_w, weight slice, view).  Output pixel (n, y, x), y < gh, x < gw, is written at
// out + base + n*s_n + y*s_h + x*s_w (+ channel).
int cgan_conv_tc(cgan_ctx* ctx, const float* in, int nviews, const long long* view_off, long long in_sw, long long in_sh,
                 long long in_sn, int n, int h, int w, int gh, int gw, int kdim, const float* wsrc, int taps_total,
                 int transpose_w,
                 int ncols, int ntaps, const int* off_h, const int* off_w, const int* wtap, const int* amap,
                 const float* bias, float* out, long long s_n, long long s_h, long long s_w, long long base, int relu,
                 const int* view_phase_of, int wimg_stride, const TcExtra* ex) {
  // ex->nphases > 1: the `ntaps` taps are the concatenation of the tap lists of nphases sub-pixel phases
  // (ex->ph_tap0[0..nphases]), phase ph writing at element offset ex->ph_base[ph] instead of `base`; one launch, grid.z
  // wimg_stride != 0: batched GEMM — image i multiplies weight slice wtap + i*wimg_stride (needs one image per tile)
  // view_phase_of: {H, W} of the tensor whose four stride-2 parity phases the views are (nullptr: all views h x w)
  EncodeTiledFn enc = get_encode();
  if (!enc) return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: cuTensorMapEncodeTiled unavailable%s", "cgan_conv_tc");
  if (ntaps > TC_MAX_TAPS || nviews > 4) return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: too many taps/views%s", "cgan_conv_tc");
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.ntaps = ntaps;
  const int kdim_pad = (kdim + TC_BK - 1) / TC_BK * TC_BK;
  p.kchunks = kdim_pad / TC_BK;
  for (int i = 0; i < ntaps; ++i) {
    p.off_h[i] = off_h[i]; p.off_w[i] = off_w[i]; p.wtap[i] = wtap[i]; p.amap[i] = amap ? amap[i] : 0;
  }
  int tiles_n;
  // the pixel grid that is tiled (gh x gw: the OUTPUT extent) may differ from the extent of the input views (h x w):
  // VALID convolutions shrink it, their taps only carry non-negative offsets
  tc_geometry(n, gh, gw, &p.bw, &p.bh, &p.bni, &p.tiles_w, &p.tiles_h, &tiles_n);
  p.rows_used = p.bw * p.bh * p.bni;
  p.img_n = n; p.img_h = gh; p.img_w = gw;
  p.relu = relu;
  p.round_a = (ex && ex->a_prerounded) ? 0 : 1;
  if (ex) {
    p.round_out = ex->round_out; p.residual = ex->residual; p.mask = ex->mask; p.mask_leak = ex->mask_leak;
  }
  p.nphases = 1;
  p.ph_tap0[0] = 0; p.ph_tap0[1] = ntaps;
  p.ph_base[0] = base;
  if (ex && ex->nphases > 1) {
    if (ex->nphases > 4) return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: more than four phases%s", "cgan_conv_tc");
    p.nphases = ex->nphases;
    for (int i = 0; i <= ex->nphases; ++i) p.ph_tap0[i] = ex->ph_tap0[i];
    for (int i = 0; i < ex->nphases; ++i) p.ph_base[i] = ex->ph_base[i];
  }
  p.wimg_stride = wimg_stride;
  if (wimg_stride != 0 && p.bni != 1)
    return cgan_fail(ctx, CGAN_ERR_UNSUPPORTED, "%s: batched GEMM needs >= 128 rows per matrix%s", "cgan_conv_tc");
  const int ncols_pad = (ncols + 31) / 32 * 32;
  p.bn = tc_pick_bn_occupancy(ncols_pad, (long long)p.tiles_w * p.tiles_h * tiles_n, ctx->num_sms);
  p.cout = ncols;
  p.s_n = s_n; p.s_h = s_h; p.s_w = s_w; p.base = base;
  p.out = out;
  p.bias = bias;

  float* wt = (ex && ex->wprep) ? const_cast<float*>(ex->wprep) : nullptr;
  if (!wt) {
    int rc = cgan_tc_prep_weights(ctx, wsrc, taps_total, transpose_w, ncols, kdim, &wt);
    if (rc) return rc;
  }

  // ---- halo variant: three taps of a kernel column share one (bh+2)-row activation box --------------------------------
  // Measured (round 2, profiles/r2_microbench.txt): with a pre-rounded operand the per-tap kernel is bound by the
  // shared-memory pipe (TMA fills + UMMA operand reads), not by the L2 feed, and the halo variant (one CTA per SM) is no
  // faster (256 -> 256) or slower (128 -> 128, which runs two per-tap CTAs per SM); it wins 8 % when the operand still
  // has to be rounded in shared memory (half the rounding work).  CGAN_OPT_TC_HALO = 2 forces it everywhere (tests).
  const bool halo_wanted = ctx->tc_halo == 2 || (ctx->tc_halo == 1 && p.round_a && ncols_pad >= 256);
  if (halo_wanted && p.nphases == 1 && nviews == 1 && wimg_stride == 0 && ntaps == 9 && gh == h && gw == w && !view_phase_of) {
    int hbw = 0, hbh = 0;
    if (w % 32 == 0) { hbw = 32; hbh = 4; } else if (w == 16) { hbw = 16; hbh = 8; }
    // group the taps by horizontal offset; each group must be three vertically consecutive taps
    int gw_off[4], gh0[4], gcnt[4] = {0, 0, 0, 0}, gtap[4][4], ng = 0;
    bool ok = hbw != 0 && h % hbh == 0 && h >= hbh;
    for (int i = 0; ok && i < ntaps; ++i) {
      int g = -1;
      for (int j = 0; j < ng; ++j)
        if (gw_off[j] == off_w[i]) g = j;
      if (g < 0) {
        if (ng == 3) { ok = false; break; }
        g = ng++; gw_off[g] = off_w[i]; gh0[g] = off_h[i];
      }
      if (gcnt[g] == 3) { ok = false; break; }
      if (off_h[i] < gh0[g]) gh0[g] = off_h[i];
      gtap[g][gcnt[g]++] = i;
    }
    ok = ok && ng == 3;
    for (int g = 0; ok && g < ng; ++g) {
      if (gcnt[g] != 3) { ok = false; break; }
      int ordered[3] = {-1, -1, -1};
      for (int j = 0; j < 3; ++j) {
        int dh = off_h[gtap[g][j]] - gh0[g];
        if (dh < 0 || dh > 2 || ordered[dh] >= 0) { ok = false; break; }
        ordered[dh] = wtap[gtap[g][j]];
      }
      for (int j = 0; ok && j < 3; ++j) p.h_wtap[g][j] = ordered[j];
      p.h_off_w[g] = gw_off[g]; p.h_off_h0[g] = gh0[g];
    }
    if (ok) {
      p.hg = 3; p.hnv = 3;
      p.bw = hbw; p.bh = hbh; p.bni = 1;
      p.tiles_w = w / hbw; p.tiles_h = h / hbh;
      const long long tiles_total = (long long)p.tiles_w * p.tiles_h * n;
      p.rows_used = 128;
      p.bn = tc_pick_bn_occupancy(ncols_pad, tiles_total, ctx->num_sms);
      const int ncol_tiles = ncols_pad / p.bn;
      p.a_box_bytes = (hbh + 2) * hbw * 128;
      p.a_halo_bytes = (p.a_box_bytes + 1023) / 1024 * 1024;
      const int b_bytes = p.bn * TC_BK * 4;
      // pixel tiles per CTA (they share every weight tile): as many as the 512 TMEM columns hold, while two waves of CTAs
      // remain and the weight ring keeps >= 4 stages (a k-block of mt tiles is ~mt*bn/2 clocks of MMA; the ring has to
      // cover the L2 latency of ~2-4 k-blocks).  The activation ring has two stages, each good for three k-blocks.
      const int budget = 227 * 1024 - 1024 - 512;
      const int mt_cap = ctx->tc_mt_max >= 2 ? 4 : 1;
      p.sa_stages = 2;
      p.mt = 1;
      for (int m = mt_cap; m >= 2; --m) {
        if (m * p.bn > 512 || tiles_total * ncol_tiles < 2ll * m * ctx->num_sms) continue;
        if ((budget - p.sa_stages * m * p.a_halo_bytes) / b_bytes < 4) continue;
        p.mt = m;
        break;
      }
      p.sb_stages = (budget - p.sa_stages * p.mt * p.a_halo_bytes) / b_bytes;
      if (p.sb_stages > 8) p.sb_stages = 8;
      ok = p.sb_stages >= 2 && (p.a_box_bytes / 16) % (32 * TC_RWARPS) == 0;
      if (ok) {
        p.tiles_total = (int)tiles_total;
        p.tmem_cols = 32;
        while (p.tmem_cols < p.mt * p.bn) p.tmem_cols *= 2;
        CUtensorMap tm_a, tm_bh;
        if (!make_act_map(&tm_a, in + view_off[0], kdim, w, h, n, in_sw, in_sh, in_sn, hbw, hbh + 2, 1))
          return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled(A halo) failed%s", "cgan_conv_tc");
        cuuint64_t dims[3] = {(cuuint64_t)kdim_pad, (cuuint64_t)ncols_pad, (cuuint64_t)taps_total};
        cuuint64_t strides[2] = {(cuuint64_t)kdim_pad * 4, (cuuint64_t)ncols_pad * kdim_pad * 4};
        cuuint32_t box[3] = {TC_BK, (cuuint32_t)p.bn, 1};
        cuuint32_t es[3] = {1, 1, 1};
        if (enc(&tm_bh, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, wt, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
          return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled(B) failed%s", "cgan_conv_tc");
        size_t smem = (size_t)p.sa_stages * p.mt * p.a_halo_bytes + (size_t)p.sb_stages * b_bytes + 1024 + 512;
        static bool halo_attr_set = false;
        if (!halo_attr_set) {
          CGAN_CUDA(ctx, cudaFuncSetAttribute(conv_tc_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
          halo_attr_set = true;
        }
        dim3 grid((unsigned)((tiles_total + p.mt - 1) / p.mt), (unsigned)ncol_tiles);
        conv_tc_halo_kernel<<<grid, TC_THREADS, smem, ctx->stream>>>(tm_a, tm_bh, p);
        CGAN_LAUNCHED(ctx);
        return CGAN_OK;
      }
    }
    // not eligible after all: restore the standard geometry
    tc_geometry(n, gh, gw, &p.bw, &p.bh, &p.bni, &p.tiles_w, &p.tiles_h, &tiles_n);
    p.rows_used = p.bw * p.bh * p.bni;
    p.bn = tc_pick_bn_occupancy(ncols_pad, (long long)p.tiles_w * p.tiles_h * tiles_n, ctx->num_sms);
    p.hg = p.hnv = 0;
  }

  AMaps tm_as;
  CUtensorMap tm_b;
  memset(&tm_as, 0, sizeof(tm_as));
  for (int v = 0; v < 4; ++v) {
    int vv = v < nviews ? v : 0;
    // stride-2 phase views of an odd-sized tensor differ in extent: rows 2r+a < H  =>  (H - a + 1) / 2 rows in phase a
    int vh = h, vw = w;
    if (nviews == 4 && view_phase_of) { vh = (view_phase_of[0] - (vv >> 1) + 1) / 2; vw = (view_phase_of[1] - (vv & 1) + 1) / 2; }
    if (vh < 1 || vw < 1) { vh = h; vw = w; vv = 0; }
    if (!make_act_map(&tm_as.m[v], in + view_off[vv], kdim, vw, vh, n, in_sw, in_sh, in_sn, p.bw, p.bh, p.bni))
      return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled(A) failed%s", "cgan_conv_tc");
  }
  {
    cuuint64_t dims[3] = {(cuuint64_t)kdim_pad, (cuuint64_t)ncols_pad, (cuuint64_t)taps_total};
    cuuint64_t strides[2] = {(cuuint64_t)kdim_pad * 4, (cuuint64_t)ncols_pad * kdim_pad * 4};
    cuuint32_t box[3] = {TC_BK, (cuuint32_t)p.bn, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(&tm_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, wt, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return cgan_fail(ctx, CGAN_ERR_CUDA, "%s: cuTensorMapEncodeTiled(B) failed%s", "cgan_conv_tc");
  }

  // Two CTAs per SM (each owns 256 of the 512 TMEM columns): one CTA's epilogue and prologue overlap the other's main
  // loop, which matters for the short-K convolutions (3x3x128: 36 k-blocks).  ~110 KB of smem each.
  // Pixel tiles per CTA: with mt = 2 the weight tile is fetched once for 256 pixels, which cuts the L2->SM bytes per MMA by
  // a third (bn = 256: 96 -> 64 B/clk/SM against a ~43 B/clk/SM L2 budget).  bn = 256 then fills the TMEM (one CTA per SM),
  // bn <= 128 keeps two CTAs per SM.  Only when enough CTAs remain to fill the machine.
  const long long tiles_total = (long long)p.tiles_w * p.tiles_h * tiles_n;
  const int ncol_tiles = ncols_pad / p.bn;
  p.tiles_total = (int)tiles_total;
  p.mt = 1;
  if (ctx->tc_mt_max >= 2 && tiles_total * ncol_tiles * p.nphases >= 4ll * ctx->num_sms &&
      (wimg_stride == 0 || (p.tiles_w * p.tiles_h) % 2 == 0))
    p.mt = 2;
  const bool two_ctas = p.mt * p.bn <= 256;
  const size_t stage_bytes = (size_t)p.mt * TC_A_BYTES + (size_t)p.bn * TC_BK * 4;
  p.stages = (int)(((two_ctas ? 110 : 220) * 1024) / stage_bytes);
  if (p.stages > TC_MAX_STAGES) p.stages = TC_MAX_STAGES;
  if (p.stages < 2) p.stages = 2;
  p.tmem_cols = 32;
  while (p.tmem_cols < p.mt * p.bn) p.tmem_cols *= 2;
  size_t smem = (size_t)p.stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/;
  static bool attr_set = false;
  if (!attr_set) {
    CGAN_CUDA(ctx, cudaFuncSetAttribute(conv_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    attr_set = true;
  }
  dim3 grid((unsigned)((tiles_total + p.mt - 1) / p.mt), (unsigned)ncol_tiles, (unsigned)p.nphases);
  conv_tc_kernel<<<grid, TC_THREADS, smem, ctx->stream>>>(tm_as, tm_b, p);
  CGAN_LAUNCHED(ctx);
  return CGAN_OK;
}
