// Forward filter / backward smoother for DENSE or WIDE-BAND "move" kernels on the tensor cores.
//
// Replaces reference poor_man_gplvm/decoder.py:151-198 and :200-332 for the transitions that
// gp_kernel.py:61-66 (custom_transition_kernel) and :14-20 with a large movement_variance produce: a K x K
// matrix whose per-bin mat-vec (4 K^2 flop per bin and pass) dominates everything else (BASELINE.json
// configs[4]: K = 2000).  A chain's mat-vec is memory/latency-bound on CUDA cores; S chains advancing in
// LOCKSTEP turn the S mat-vecs of one time step into ONE GEMM
//
//        D[c, x'] = sum_x U[c, x] * P[x, x']            [S x K] . [K x K]
//
// that runs on tcgen05 (kind::f16, TMA-fed, fp32 accumulation in TMEM).  Both operands are carried as two
// fp16 pieces (hi + lo = 22 significant bits) under exact power-of-two scales -- the chain message is
// renormalised every step, so a per-row scale keeps it inside the fp16 range -- and a step issues the three
// products hi*hi + hi*lo + lo*hi.  Everything else of the recursion (likelihood factor, rank-1 jump term,
// normaliser, outputs, seam / warm-start messages) is a per-chain row operation in `dense_*_update_kernel`
// (one CTA per chain, fp32).  One pass = hmax + chunk_len steps of [GEMM, update], enqueued by one C call.
//
// Chain / warm-up / seam conventions are those of pmg_forward / pmg_backward (pmg_scan.cu), mode 0 only:
// repairs of individual chains (modes 1, 2) go through the general kernels.
#include <cuda_fp16.h>

#include "pmg_chain.cuh"
#include "pmg_tc.cuh"

namespace pmg {
using namespace tc;

constexpr int DS_BM = 128;                       // chains per accumulator tile (TMEM lanes)
constexpr int DS_BK = 64;                        // fp16 elements per K block = one 128-byte swizzle row
constexpr int DS_A_BYTES = DS_BM * DS_BK * 2;    // 16 KB per piece
constexpr int DS_EPI_WARPS = 8;                  // epilogue warps: 4 TMEM lane quarters x 2 column halves
constexpr int DS_EPI_COLS = 128;                 // accumulator columns an epilogue thread keeps in registers
constexpr int DS_THREADS = 32 * (4 + DS_EPI_WARPS);   // GEMM: warp 0 TMA, 1 MMA, 2 TMEM alloc, 4-11 epilogue
constexpr int DS_MAX_NT = 16;                    // column tiles (K <= 4096)
constexpr int DS_UPD_THREADS = 256;
constexpr float kDsPieceScale = 16384.f;         // 2^14: pieces of values in [0, 2) stay below the fp16 maximum

struct DenseGeo {
  int K, Kk, Kn, BN, n_ntiles;
};

static DenseGeo dense_geo(int K) {
  DenseGeo g;
  g.K = K;
  g.Kk = (K + DS_BK - 1) / DS_BK * DS_BK;        // reduction length (columns of both operands)
  g.n_ntiles = (K + 255) / 256;
  int bn = (K + g.n_ntiles - 1) / g.n_ntiles;
  g.BN = (bn + 15) / 16 * 16;                    // accumulator columns per tile
  g.Kn = g.n_ntiles * g.BN;                      // rows of the right-hand operand = columns of D
  return g;
}

struct DenseGemmParams {
  int n_mtiles, n_ntiles, BN, stages;
  int kb_per_chunk;                              // K blocks accumulated in TMEM before they are drained (see the kernel)
  int col_split;                                 // columns [0, col_split) / [col_split, BN) of a tile per epilogue half
  int a_rows, b_rows;                            // rows per piece of the two operands
  int kb_lo[DS_MAX_NT], kb_hi[DS_MAX_NT];        // K blocks that hold non-zeros of a column tile (band structure)
  uint32_t idesc, tmem_cols;
  float* D;
  int64_t ldd;
};

// D[m, n] = sum_k (Ah + Al)[m,k] * (Bh + Bl)[n,k] - Al*Bl, persistent over (row tile, column tile) units.
//
// Accumulation.  The tensor core adds into its fp32 accumulator with truncation, and every tcgen05.mma on the same
// TMEM accumulator loses a fraction of an ulp of the RUNNING sum: measured here, a K = 2000 reduction (384 MMAs into one
// accumulator) comes out 1e-4 low, linearly in the number of MMAs -- systematic, because all terms are positive
// (see Ootomo & Yokota, "Recovering single precision accuracy from Tensor Cores", for the same effect on mma.sync).
// So an accumulator only ever holds a CHUNK of `kb_per_chunk` K blocks (12 MMAs per block), two accumulators
// alternate, and the eight epilogue warps drain each finished chunk into fp32 registers with round-to-nearest adds
// while the next chunk's MMAs run; the registers hold the tile until it is stored.
__global__ void __launch_bounds__(DS_THREADS, 1)
dense_step_gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                       const DenseGemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = p.BN;
  const uint32_t b_bytes = (uint32_t)BN * DS_BK * 2;
  const uint32_t stage_bytes = 2 * DS_A_BYTES + 2 * b_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 32 * DS_EPI_WARPS); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); }
  if (warp == 2) { tmem_alloc(tmem_slot, p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_tiles = p.n_mtiles * p.n_ntiles;
  const int cpk = p.kb_per_chunk;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        // consecutive CTAs share a row tile (the small operand) and walk the column tiles
        const int mt = tile / p.n_ntiles, nt = tile % p.n_ntiles;
        for (int kb = p.kb_lo[nt]; kb < p.kb_hi[nt]; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + (size_t)stage * stage_bytes;
          mbar_arrive_expect_tx(&full[stage], stage_bytes);
          tma_load_2d(sA, &tmA, &full[stage], kb * DS_BK, mt * DS_BM);
          tma_load_2d(sA + DS_A_BYTES, &tmA, &full[stage], kb * DS_BK, p.a_rows + mt * DS_BM);
          tma_load_2d(sA + 2 * DS_A_BYTES, &tmB, &full[stage], kb * DS_BK, nt * BN);
          tma_load_2d(sA + 2 * DS_A_BYTES + b_bytes, &tmB, &full[stage], kb * DS_BK, p.b_rows + nt * BN);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;        // it: chunks issued so far (across tiles)
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_ntiles;
        for (int kb0 = p.kb_lo[nt]; kb0 < p.kb_hi[nt]; kb0 += cpk, ++it) {
          const int buf = it & 1;
          const uint32_t acc_phase = (it >> 1) & 1;
          mbar_wait(&tempty[buf], acc_phase ^ 1);
          tc_fence_after();
          const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
          uint32_t acc = 0;
          const int kb1 = kb0 + cpk < p.kb_hi[nt] ? kb0 + cpk : p.kb_hi[nt];
          for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(&full[stage], phase);
            tc_fence_after();
            const uint32_t sAh = smem_u32(smem + (size_t)stage * stage_bytes);
            const uint32_t sAl = sAh + DS_A_BYTES;
            const uint32_t sBh = sAh + 2 * DS_A_BYTES;
            const uint32_t sBl = sBh + b_bytes;
#pragma unroll
            for (int k = 0; k < DS_BK / 16; ++k) {
              const uint64_t ah = make_smem_desc(sAh + k * 32, 16, 1024);
              const uint64_t al = make_smem_desc(sAl + k * 32, 16, 1024);
              const uint64_t bh = make_smem_desc(sBh + k * 32, 16, 1024);
              const uint64_t bl = make_smem_desc(sBl + k * 32, 16, 1024);
              // small products first: they are added while the accumulator is still small
              mma_f16_ss(d_tmem, ah, bl, p.idesc, acc);
              acc = 1;
              mma_f16_ss(d_tmem, al, bh, p.idesc, 1);
              mma_f16_ss(d_tmem, ah, bh, p.idesc, 1);
            }
            mma_commit(&empty[stage]);
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          mma_commit(&tfull[buf]);
        }
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;            // column half this warp drains
    const int c_lo = half == 0 ? 0 : p.col_split;
    const int c_hi = half == 0 ? p.col_split : BN;
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const int mt = tile / p.n_ntiles, nt = tile % p.n_ntiles;
      float sum[DS_EPI_COLS];
#pragma unroll
      for (int j = 0; j < DS_EPI_COLS; ++j) sum[j] = 0.f;
      for (int kb0 = p.kb_lo[nt]; kb0 < p.kb_hi[nt]; kb0 += cpk, ++it) {
        const int buf = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tfull[buf], acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + c_lo);
#pragma unroll
        for (int g = 0; g < DS_EPI_COLS / 16; ++g) {
          if (c_lo + g * 16 < c_hi) {            // BN and col_split are multiples of 16: whole loads only
            uint32_t r[16];
            tmem_ld_x16(taddr + g * 16, r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) sum[g * 16 + j] += __uint_as_float(r[j]);
          }
        }
        tc_fence_before();
        mbar_arrive(&tempty[buf]);
      }
      float* orow = p.D + (size_t)(mt * DS_BM + q * 32 + lane) * p.ldd + (size_t)nt * BN + c_lo;
#pragma unroll
      for (int g = 0; g < DS_EPI_COLS / 32; ++g) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (c_lo + g * 32 + j < c_hi)          // BN and col_split are multiples of 8: float4 groups never straddle
            *reinterpret_cast<float4*>(orow + g * 32 + j) =
                make_float4(sum[g * 32 + j], sum[g * 32 + j + 1], sum[g * 32 + j + 2], sum[g * 32 + j + 3]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, p.tmem_cols); }
}

// ---------------------------------------------------------------------------------------------
// per-chain row operations
// ---------------------------------------------------------------------------------------------
// the chain plan (mode 0) and the lockstep operands
struct DenseChains : ScanCommon {
  int hmax;                // warm-up steps of the pass: per-chain warm-ups are capped at hmax
  const float* D;          // GEMM result [S_pad, ldd]
  int64_t ldd;
  __half* U16;             // left-hand operand of the next step: [2][S_pad][Kk] fp16 pieces
  int64_t ldu;
  int64_t u_piece;         // elements between the hi and the lo piece
  float* state;            // [n_chain][4]
};

struct DenseFwdParams {
  DenseChains c;
  const float* carry_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  float* alpha;
  float* lmr;
  float* halo_state;
};

struct DenseBwdParams {
  DenseChains c;
  const float* alpha;
  const float* beta_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  float* gamma;
  float* gamma_lat;
  __half* gamma16;
  int64_t ldg;
  float* dyn_marg;
  float* r_out;
  float* r_scratch;        // [n_chain][2][K]: r of the bin handled last (normalised by its own step only)
  float* tw_partial;
  float* beta_halo;
  float* beta_end;
};

// block-wide reductions over DS_UPD_THREADS threads; `slot` selects a private scratch row (no reuse hazard
// between the reductions of one step)
__device__ __forceinline__ float block_max(float v, float* red, int slot) {
  v = warp_max(v);
  float* r = red + slot * 16;
  if ((threadIdx.x & 31) == 0) r[threadIdx.x >> 5] = v;
  __syncthreads();
  float m = r[0];
#pragma unroll
  for (int w = 1; w < DS_UPD_THREADS / 32; ++w) m = fmaxf(m, r[w]);
  return m;
}
__device__ __forceinline__ void block_sum2(float& a, float& b, float* red, int slot) {
  a = warp_sum(a); b = warp_sum(b);
  float* r = red + slot * 16;
  if ((threadIdx.x & 31) == 0) { r[threadIdx.x >> 5] = a; r[8 + (threadIdx.x >> 5)] = b; }
  __syncthreads();
  float sa = 0.f, sb = 0.f;
#pragma unroll
  for (int w = 0; w < DS_UPD_THREADS / 32; ++w) { sa += r[w]; sb += r[8 + w]; }
  a = sa; b = sb;
}

// exact power-of-two scale that brings `vmax` into [2^14, 2^15): returns the scale, *inv_scale its reciprocal
// (exponents beyond +-100 are clamped: a renormalised message never gets there)
__device__ __forceinline__ float piece_scale(float vmax, float* inv_scale) {
  if (!(vmax > 0.f) || !(vmax < 3.0e38f)) { *inv_scale = 1.f / kDsPieceScale; return kDsPieceScale; }
  int e = (int)((__float_as_uint(vmax) >> 23) & 0xff) - 127;             // floor(log2 vmax)
  e = e < -100 ? -100 : (e > 100 ? 100 : e);
  const float s = __uint_as_float((uint32_t)(127 + 14 - e) << 23);        // 2^(14 - e)
  *inv_scale = __uint_as_float((uint32_t)(127 - 14 + e) << 23);
  return s;
}
__device__ __forceinline__ void store_pieces(__half* hi, __half* lo, float v) {
  const __half h = __float2half_rn(v);
  *hi = h;
  *lo = __float2half_rn(v - __half2float(h));
}

// One step of every chain's forward recursion (reference decoder.py:151-172).  step -1 only initialises.
template <int EPT>
__global__ void __launch_bounds__(DS_UPD_THREADS) dense_fwd_update_kernel(const DenseFwdParams p, const int step) {
  __shared__ float red[48];
  const DenseChains& c = p.c;
  const int s = blockIdx.x;
  const int64_t t_begin = c.core_begin + (int64_t)s * c.chunk_len;
  int64_t t_end = t_begin + c.chunk_len;
  if (t_end > c.core_end) t_end = c.core_end;
  if (t_begin >= t_end) return;
  const ChainRange cr{s, t_begin, t_end};
  const int K = c.tr.K;
  int64_t t0;
  const float* src = fwd_start<false>(c, cr, p, t0, K, c.hmax);
  const int j = step - (c.hmax - (int)(t_begin - t0));
  if (j < -1) return;
  const int64_t t = t0 + j;
  if (t >= t_end) return;
  const float invK = 1.f / (float)K;
  float* st = c.state + (size_t)s * 4;
  __half* uh = c.U16 + (size_t)s * c.ldu;
  __half* ul = uh + c.u_piece;

  float a0[EPT], a1[EPT];
  float S0, S1;
  if (j == -1) {
    // ---- initial carry: exact start (carry_in or uniform) or the warm-start message; normalised to unit sum
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      const bool ok = x < K;
      a0[e] = ok ? (src ? src[x] : 0.5f * invK) : 0.f;
      a1[e] = ok ? (src ? src[K + x] : 0.5f * invK) : 0.f;
      s0 += a0[e]; s1 += a1[e];
    }
    block_sum2(s0, s1, red, 0);
    if (!(s0 + s1 > 0.f) || !(s0 + s1 < 3.0e38f)) {          // unusable message: uniform
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const bool ok = threadIdx.x + e * DS_UPD_THREADS < K;
        a0[e] = ok ? 0.5f * invK : 0.f; a1[e] = a0[e];
      }
      s0 = 0.5f; s1 = 0.5f;
    }
    const float inv = 1.f / (s0 + s1);
#pragma unroll
    for (int e = 0; e < EPT; ++e) { a0[e] *= inv; a1[e] *= inv; }
    S0 = s0 * inv; S1 = s1 * inv;
  } else {
    // ---- prior (move part from the GEMM, jump part rank-1) x likelihood factor, normaliser
    const float* drow = c.D + (size_t)s * c.ldd;
    const float* lrow = c.ll + (size_t)t * c.ldll;
    const float uscale = st[2];
    const float p1 = (c.tr.M01 * st[0] + c.tr.M11 * st[1]) * invK;
    float L[EPT];
    float m = -INFINITY;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      L[e] = x < K ? lrow[x] : -INFINITY;
      m = fmaxf(m, L[e]);
    }
    m = block_max(m, red, 0);
    const float sc2 = c.scale * 1.4426950408889634f;
    const float msc = m * sc2;
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      const float Lx = x < K ? exp2f(fmaf(L[e], sc2, -msc)) : 0.f;
      const float d = x < K ? drow[x] * uscale : 0.f;
      a0[e] = d * Lx;
      a1[e] = p1 * Lx;
      s0 += a0[e]; s1 += a1[e];
    }
    block_sum2(s0, s1, red, 1);
    const float cn = s0 + s1;
    const float inv = 1.f / cn;
#pragma unroll
    for (int e = 0; e < EPT; ++e) { a0[e] *= inv; a1[e] *= inv; }
    S0 = s0 * inv; S1 = s1 * inv;
    if (t >= t_begin) {
      float* o = p.alpha + (size_t)t * 2 * K;
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int x = threadIdx.x + e * DS_UPD_THREADS;
        if (x < K) { o[x] = a0[e]; o[K + x] = a1[e]; }
      }
      if (threadIdx.x == 0) p.lmr[t] = logf(cn) + c.scale * m;
    } else if (t == t_begin - 1 && p.halo_state) {
      float* o = p.halo_state + (size_t)s * 2 * K;
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int x = threadIdx.x + e * DS_UPD_THREADS;
        if (x < K) { o[x] = a0[e]; o[K + x] = a1[e]; }
      }
    }
    if (p.warm_out && t == t_end - halo_next_of(c, s + 1) - 1 && (s + 1 < c.n_chain || !c.right_exact)) {
      float* o = p.warm_out + (size_t)(s + 1) * 2 * K;
#pragma unroll
      for (int e = 0; e < EPT; ++e) {
        const int x = threadIdx.x + e * DS_UPD_THREADS;
        if (x < K) { o[x] = a0[e]; o[K + x] = a1[e]; }
      }
    }
  }
  // ---- left-hand operand of the next step: u = M00 alpha0 + M10 alpha1 as two scaled fp16 pieces
  float umax = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e) { a0[e] = fmaf(c.tr.M00, a0[e], c.tr.M10 * a1[e]); umax = fmaxf(umax, a0[e]); }
  umax = block_max(umax, red, 2);
  float inv_scale;
  const float us = piece_scale(umax, &inv_scale);
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int x = threadIdx.x + e * DS_UPD_THREADS;
    if (x < K) store_pieces(uh + x, ul + x, a0[e] * us);
  }
  if (threadIdx.x == 0) { st[0] = S0; st[1] = S1; st[2] = inv_scale * (1.f / kDsPieceScale); }
}

// One step of every chain's backward recursion (reference decoder.py:200-256), bins in descending order.
template <int EPT>
__global__ void __launch_bounds__(DS_UPD_THREADS) dense_bwd_update_kernel(const DenseBwdParams p, const int step) {
  __shared__ float red[48];
  const DenseChains& c = p.c;
  const int s = blockIdx.x;
  const int64_t t_begin = c.core_begin + (int64_t)s * c.chunk_len;
  int64_t t_end = t_begin + c.chunk_len;
  if (t_end > c.core_end) t_end = c.core_end;
  if (t_begin >= t_end) return;
  const ChainRange cr{s, t_begin, t_end};
  const int K = c.tr.K;
  int64_t t_hi;
  const float* init = bwd_start<false>(c, cr, p, t_hi, K, c.hmax);
  const int j = step - (c.hmax - (int)(t_hi - (t_end - 1)));
  if (j < 0) return;
  const int64_t t = t_hi - j;
  if (t < t_begin) return;
  const float invK = 1.f / (float)K;
  float* st = c.state + (size_t)s * 4;

  // ---- unnormalised beta_t
  float b0[EPT], b1[EPT];
  if (j == 0) {
    float sb = 0.f, dummy = 0.f;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      const bool ok = x < K;
      b0[e] = ok ? (init ? init[x] : 1.f) : 0.f;
      b1[e] = ok ? (init ? init[K + x] : 1.f) : 0.f;
      sb += b0[e] + b1[e];
    }
    block_sum2(sb, dummy, red, 0);
    if (!(sb > 0.f) || !(sb < 3.0e38f)) {                    // unusable message: all ones
#pragma unroll
      for (int e = 0; e < EPT; ++e) { b0[e] = (threadIdx.x + e * DS_UPD_THREADS < K) ? 1.f : 0.f; b1[e] = b0[e]; }
    }
  } else {
    const float* drow = c.D + (size_t)s * c.ldd;
    const float w1 = st[0], rscale = st[1];
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      const float w0 = x < K ? drow[x] * rscale : 0.f;
      b0[e] = x < K ? fmaf(c.tr.M00, w0, c.tr.M01 * w1) : 0.f;
      b1[e] = x < K ? fmaf(c.tr.M10, w0, c.tr.M11 * w1) : 0.f;
    }
  }
  // ---- likelihood factor, normaliser, posterior
  const float* lrow = c.ll + (size_t)t * c.ldll;
  float L[EPT];
  float m = -INFINITY;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int x = threadIdx.x + e * DS_UPD_THREADS;
    L[e] = x < K ? lrow[x] : -INFINITY;
    m = fmaxf(m, L[e]);
  }
  m = block_max(m, red, 1);
  const float sc2 = c.scale * 1.4426950408889634f;
  const float msc = m * sc2;
  const bool use_alpha = t <= t_end;
  float g0[EPT], g1[EPT];
  float s0 = 0.f, s1 = 0.f;
  if (use_alpha) {
    const float* arow = p.alpha + (size_t)t * 2 * K;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      g0[e] = x < K ? arow[x] * b0[e] : 0.f;
      g1[e] = x < K ? arow[K + x] * b1[e] : 0.f;
      s0 += g0[e]; s1 += g1[e];
    }
  } else {
#pragma unroll
    for (int e = 0; e < EPT; ++e) { g0[e] = 0.f; g1[e] = 0.f; s0 += b0[e]; s1 += b1[e]; }
  }
  block_sum2(s0, s1, red, 2);
  const float inv = 1.f / (s0 + s1);

  if (t < t_end) {
    float* g = p.gamma ? p.gamma + (size_t)t * 2 * K : nullptr;
    float* gl = p.gamma_lat ? p.gamma_lat + (size_t)t * K : nullptr;
    __half* gh = p.gamma16 ? p.gamma16 + (size_t)t * p.ldg : nullptr;
    __half* glo = p.gamma16 ? p.gamma16 + ((size_t)c.T + t) * p.ldg : nullptr;
    float* tw = p.tw_partial ? p.tw_partial + (size_t)s * K : nullptr;
    const bool first = t == t_end - 1;
    const float* rs = (p.r_out && j > 0) ? p.r_scratch + (size_t)s * 2 * K : nullptr;
    float* ro = rs ? p.r_out + (size_t)(t + 1) * 2 * K : nullptr;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      if (x < K) {
        const float ga = g0[e] * inv, gb = g1[e] * inv, gs = ga + gb;
        if (g) { g[x] = ga; g[K + x] = gb; }
        if (gl) gl[x] = gs;
        if (gh) store_pieces(gh + x, glo + x, gs);
        if (tw) tw[x] = first ? gs : tw[x] + gs;
        if (ro) { ro[x] = rs[x] * inv; ro[K + x] = rs[K + x] * inv; }      // r_{t+1} / z_t
      }
    }
    if (p.dyn_marg && threadIdx.x == 0) { p.dyn_marg[2 * t] = s0 * inv; p.dyn_marg[2 * t + 1] = s1 * inv; }
  } else if (t == t_end && p.beta_halo) {
    float* o = p.beta_halo + (size_t)s * 2 * K;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      if (x < K) { o[x] = b0[e] * inv; o[K + x] = b1[e] * inv; }
    }
  }
  if (t == t_begin && p.beta_end) {
    float* o = p.beta_end + (size_t)s * 2 * K;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      if (x < K) { o[x] = b0[e] * inv; o[K + x] = b1[e] * inv; }
    }
  }
  if (p.warm_out && t == t_begin + halo_next_of(c, s - 1) - 1 && (s >= 1 || !c.left_exact)) {
    float* o = p.warm_out + ((int64_t)s - 1) * 2 * K;
#pragma unroll
    for (int e = 0; e < EPT; ++e) {
      const int x = threadIdx.x + e * DS_UPD_THREADS;
      if (x < K) { o[x] = b0[e] * inv; o[K + x] = b1[e] * inv; }
    }
  }
  // ---- r_t = L_t * beta_t (normalised by this step): its move part is the next step's left-hand operand,
  //      its jump part enters through the scalar w1 = sum_x r_t[1,x] / K
  float r1s = 0.f, rmax = 0.f;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int x = threadIdx.x + e * DS_UPD_THREADS;
    const float Lx = x < K ? exp2f(fmaf(L[e], sc2, -msc)) * inv : 0.f;
    b0[e] *= Lx; b1[e] *= Lx;
    r1s += b1[e];
    rmax = fmaxf(rmax, b0[e]);
  }
  float dummy = 0.f;
  block_sum2(r1s, dummy, red, 0);          // slot 0 was last read before the block_max above: safe to reuse
  rmax = block_max(rmax, red, 1);
  float inv_scale;
  const float rsq = piece_scale(rmax, &inv_scale);
  __half* uh = c.U16 + (size_t)s * c.ldu;
  __half* ul = uh + c.u_piece;
  float* rsc = p.r_out ? p.r_scratch + (size_t)s * 2 * K : nullptr;
#pragma unroll
  for (int e = 0; e < EPT; ++e) {
    const int x = threadIdx.x + e * DS_UPD_THREADS;
    if (x < K) {
      store_pieces(uh + x, ul + x, b0[e] * rsq);
      if (rsc) { rsc[x] = b0[e]; rsc[K + x] = b1[e]; }
    }
  }
  if (threadIdx.x == 0) { st[0] = r1s * invK; st[1] = inv_scale * (1.f / kDsPieceScale); }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct DenseWorkspace {
  __half* U16;
  float* D;
  float* state;
  float* r_scratch;
  int S_pad;
  size_t bytes;
};

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

static DenseWorkspace dense_workspace(void* base, int n_chain, const DenseGeo& g) {
  DenseWorkspace w;
  w.S_pad = (n_chain + DS_BM - 1) / DS_BM * DS_BM;
  size_t off = 0;
  char* b = (char*)base;
  w.U16 = (__half*)(b + off); off += align256((size_t)2 * w.S_pad * g.Kk * sizeof(__half));
  w.D = (float*)(b + off); off += align256((size_t)w.S_pad * g.Kn * sizeof(float));
  w.state = (float*)(b + off); off += align256((size_t)n_chain * 4 * sizeof(float));
  w.r_scratch = (float*)(b + off); off += align256((size_t)n_chain * 2 * g.K * sizeof(float));
  w.bytes = off;
  return w;
}

// validates plan, transition and operands of a lockstep pass (mode 0) and fills c; g and w receive the geometry and
// the workspace layout
static int dense_fill_chains(DenseChains& c, DenseGeo& g, DenseWorkspace& w, const pmg_scan_plan* plan,
                             const pmg_transition* tr, const void* P16, int halo_max, const float* ll, int64_t ldll,
                             void* workspace, int64_t workspace_bytes, bool fwd) {
  const int rc = fill_common(c, plan, tr, ll, ldll, 0, nullptr, 0, fwd);
  if (rc) return rc;
  if (!P16 || !workspace || halo_max < 0) return PMG_ERR_BAD_ARG;
  if (tr->K < 16 || tr->K > 256 * DS_MAX_NT) return PMG_ERR_UNSUPPORTED_SHAPE;
  if (((uintptr_t)P16 | (uintptr_t)workspace) & 255) return PMG_ERR_ALIGNMENT;
  g = dense_geo(tr->K);
  w = dense_workspace(workspace, plan->n_chain, g);
  if ((int64_t)w.bytes > workspace_bytes) return PMG_ERR_WORKSPACE;
  c.hmax = plan->halo_arr ? (halo_max > plan->halo ? halo_max : plan->halo) : plan->halo;
  c.D = w.D; c.ldd = g.Kn;
  c.U16 = w.U16; c.ldu = g.Kk; c.u_piece = (int64_t)w.S_pad * g.Kk;
  c.state = w.state;
  return PMG_OK;
}

static uint32_t ds_pow2_cols(int cols) {
  uint32_t v = 32;
  while ((int)v < cols) v <<= 1;
  return v;
}

struct DenseGemmLaunch {
  CUtensorMap tmA, tmB;
  DenseGemmParams p;
  int grid;
  size_t smem;
};

static int dense_gemm_setup(DenseGemmLaunch& L, const DenseGeo& g, const DenseWorkspace& w, const void* P16_dir,
                            const int* kb_ranges /* [n_ntiles][2] host */) {
  DenseGemmParams& p = L.p;
  p.n_mtiles = w.S_pad / DS_BM;
  p.n_ntiles = g.n_ntiles;
  p.BN = g.BN;
  p.a_rows = w.S_pad;
  p.b_rows = g.Kn;
  const int n_kb = g.Kk / DS_BK;
  for (int i = 0; i < g.n_ntiles; ++i) {
    int lo = kb_ranges ? kb_ranges[2 * i] : 0, hi = kb_ranges ? kb_ranges[2 * i + 1] : n_kb;
    if (lo < 0) lo = 0;
    if (hi > n_kb) hi = n_kb;
    if (hi <= lo) { lo = 0; hi = 1; }            // an all-zero column tile still needs one (zero) product
    p.kb_lo[i] = lo; p.kb_hi[i] = hi;
  }
  p.idesc = make_idesc_f16(DS_BM, g.BN, 0, 0, 0);
  p.kb_per_chunk = 2;
  p.col_split = (g.BN / 2 + 15) / 16 * 16;       // whole 16-column TMEM loads in both halves
  if (p.col_split > DS_EPI_COLS || g.BN - p.col_split > DS_EPI_COLS) return PMG_ERR_UNSUPPORTED_SHAPE;
  p.tmem_cols = ds_pow2_cols(2 * g.BN);
  if (p.tmem_cols > 512) return PMG_ERR_UNSUPPORTED_SHAPE;
  p.D = w.D;
  p.ldd = g.Kn;
  const size_t stage_bytes = 2 * (size_t)DS_A_BYTES + 2 * (size_t)g.BN * DS_BK * 2;
  int stages = (int)((size_t)(220 * 1024) / stage_bytes);
  if (stages > 6) stages = 6;
  if (stages < 2) return PMG_ERR_UNSUPPORTED_SHAPE;
  p.stages = stages;
  L.smem = (size_t)stages * stage_bytes + 1024 + 256;
  if (make_tmap_f16(&L.tmA, w.U16, (uint64_t)2 * w.S_pad, (uint64_t)g.Kk, (uint64_t)g.Kk, DS_BM)) return PMG_ERR_BAD_ARG;
  if (make_tmap_f16(&L.tmB, P16_dir, (uint64_t)2 * g.Kn, (uint64_t)g.Kk, (uint64_t)g.Kk, (uint32_t)g.BN)) return PMG_ERR_BAD_ARG;
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n_tiles = p.n_mtiles * p.n_ntiles;
  L.grid = n_tiles < sms ? n_tiles : sms;
  PMG_CUDA_CHECK(cudaFuncSetAttribute(dense_step_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.smem));
  return PMG_OK;
}

template <typename P, typename F>
static int dense_run(const DenseGemmLaunch& L, const P& p, int n_chain, int n_steps, F launch_update, cudaStream_t st) {
  launch_update(p, -1);
  PMG_LAUNCH_CHECK();
  for (int step = 0; step < n_steps; ++step) {
    dense_step_gemm_kernel<<<L.grid, DS_THREADS, L.smem, st>>>(L.tmA, L.tmB, L.p);
    launch_update(p, step);
  }
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

}  // namespace pmg

extern "C" int pmg_dense_scan_geometry(int K, int* Kk, int* Kn, int* BN, int* n_ntiles) {
  if (K < 16 || K > 256 * pmg::DS_MAX_NT) return PMG_ERR_UNSUPPORTED_SHAPE;
  const pmg::DenseGeo g = pmg::dense_geo(K);
  if (Kk) *Kk = g.Kk;
  if (Kn) *Kn = g.Kn;
  if (BN) *BN = g.BN;
  if (n_ntiles) *n_ntiles = g.n_ntiles;
  return PMG_OK;
}

extern "C" int64_t pmg_dense_scan_workspace_bytes(int n_chain, int K) {
  if (n_chain <= 0 || K < 16 || K > 256 * pmg::DS_MAX_NT) return 0;
  return (int64_t)pmg::dense_workspace(nullptr, n_chain, pmg::dense_geo(K)).bytes;
}

extern "C" int pmg_forward_dense(const pmg_scan_plan* plan, const pmg_transition* tr, const void* P16,
                                 const int* kb_ranges, int halo_max, const float* ll, int64_t ldll,
                                 const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                                 float* alpha, float* lmr, float* halo_state, void* workspace,
                                 int64_t workspace_bytes, pmg_stream_t stream) {
  using namespace pmg;
  DenseFwdParams p;
  DenseGeo g;
  DenseWorkspace w;
  int rc = dense_fill_chains(p.c, g, w, plan, tr, P16, halo_max, ll, ldll, workspace, workspace_bytes, true);
  if (rc) return rc;
  if (!alpha || !lmr) return PMG_ERR_BAD_ARG;
  p.carry_in = carry_in; p.warm_in = warm_in; p.warm_stride = warm_stride; p.warm_out = warm_out;
  p.alpha = alpha; p.lmr = lmr; p.halo_state = halo_state;
  DenseGemmLaunch L;
  rc = dense_gemm_setup(L, g, w, P16, kb_ranges);          // forward operand: B[x', x] = P0[x, x']
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  // padding rows / columns of the left-hand operand are never written: zero them once per pass
  PMG_CUDA_CHECK(cudaMemsetAsync(w.U16, 0, (size_t)2 * w.S_pad * g.Kk * sizeof(__half), st));
  const int n_steps = p.c.hmax + (int)plan->chunk_len;
  const int S = plan->n_chain;
  auto upd = [&](const DenseFwdParams& q, int step) {
    if (tr->K <= 4 * DS_UPD_THREADS) dense_fwd_update_kernel<4><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
    else if (tr->K <= 8 * DS_UPD_THREADS) dense_fwd_update_kernel<8><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
    else dense_fwd_update_kernel<16><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
  };
  return dense_run(L, p, S, n_steps, upd, st);
}

extern "C" int pmg_backward_dense(const pmg_scan_plan* plan, const pmg_transition* tr, const void* P16,
                                  const int* kb_ranges, int halo_max, const float* ll, int64_t ldll,
                                  const float* alpha, const float* beta_in, const float* warm_in,
                                  int64_t warm_stride, float* warm_out, float* gamma, float* gamma_lat,
                                  void* gamma16, int64_t ldg, float* dyn_marg, float* r_out, float* tw_partial,
                                  float* beta_halo, float* beta_end, void* workspace, int64_t workspace_bytes,
                                  pmg_stream_t stream) {
  using namespace pmg;
  DenseBwdParams p;
  DenseGeo g;
  DenseWorkspace w;
  int rc = dense_fill_chains(p.c, g, w, plan, tr, P16, halo_max, ll, ldll, workspace, workspace_bytes, false);
  if (rc) return rc;
  if (!alpha) return PMG_ERR_BAD_ARG;
  if (gamma16 && (ldg < tr->K || (ldg & 7))) return PMG_ERR_BAD_ARG;
  p.alpha = alpha; p.beta_in = beta_in; p.warm_in = warm_in; p.warm_stride = warm_stride; p.warm_out = warm_out;
  p.gamma = gamma; p.gamma_lat = gamma_lat; p.gamma16 = (__half*)gamma16; p.ldg = ldg;
  p.dyn_marg = dyn_marg; p.r_out = r_out; p.r_scratch = w.r_scratch; p.tw_partial = tw_partial;
  p.beta_halo = beta_halo; p.beta_end = beta_end;
  DenseGemmLaunch L;
  // backward operand: B[x, x'] = P0[x, x'] -- the second [2][Kn][Kk] block of P16
  const __half* Pb = (const __half*)P16 + (size_t)2 * g.Kn * g.Kk;
  rc = dense_gemm_setup(L, g, w, Pb, kb_ranges ? kb_ranges + 2 * g.n_ntiles : nullptr);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  PMG_CUDA_CHECK(cudaMemsetAsync(w.U16, 0, (size_t)2 * w.S_pad * g.Kk * sizeof(__half), st));
  const int n_steps = p.c.hmax + (int)plan->chunk_len;
  const int S = plan->n_chain;
  auto upd = [&](const DenseBwdParams& q, int step) {
    if (step < 0) return;                        // the backward pass initialises inside its first step
    if (tr->K <= 4 * DS_UPD_THREADS) dense_bwd_update_kernel<4><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
    else if (tr->K <= 8 * DS_UPD_THREADS) dense_bwd_update_kernel<8><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
    else dense_bwd_update_kernel<16><<<S, DS_UPD_THREADS, 0, st>>>(q, step);
  };
  return dense_run(L, p, S, n_steps, upd, st);
}
