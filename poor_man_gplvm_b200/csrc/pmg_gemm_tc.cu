// Tensor-core (tcgen05 + TMEM + TMA) GEMMs of the EM hot path.
//
//  * emission (reference poor_man_gplvm/decoder.py:30-48, :60-71):
//      ll[t,k] = sum_n y[t,n] * loglam[k,n] - lam_sum[k] - lgam[t]
//    y is stored once as fp16 (spike counts are exact in fp16 up to 2048); loglam is split into
//    two fp16 pieces (hi + lo = 22 significant bits), both K-major, so the product needs two
//    kind::f16 MMAs per K step accumulating in fp32 in TMEM.
//  * time reduction (reference fit_tuning_helper.py:28-42):
//      yw[k,n] = sum_t gamma[t,k] * y[t,n]
//    both operands have time as the slow axis (MN-major UMMA operands); gamma arrives as two
//    fp16 pieces written by the backward scan.
//
// Persistent, warp-specialised CTAs: warp 0 = TMA producer, warp 1 = MMA issuer (one thread),
// warp 2 = TMEM allocator, warps 4-7 = epilogue (TMEM -> registers -> global).
#include "pmg_common.cuh"
#include "pmg_tc.cuh"
#include <cuda_bf16.h>

namespace pmg {

using namespace tc;

constexpr int TC_BM = 128;        // rows of the accumulator tile (TMEM lanes)
constexpr int TC_BK = 64;         // fp16 elements per K block = one 128-byte swizzle row
constexpr int TC_THREADS = 256;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;   // 16 KB

// ---------------------------------------------------------------------------------------------
// conversions
// ---------------------------------------------------------------------------------------------
__global__ void counts_to_f16_kernel(int64_t T, int N, const float* __restrict__ y, int64_t ldy,
                                     __half* __restrict__ y16, int64_t ld16, int* __restrict__ inexact) {
  const int64_t total = T * ld16;
  int bad = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / ld16;
    const int n = (int)(i - t * ld16);
    float v = 0.f;
    if (n < N) v = y[(size_t)t * ldy + n];
    const __half h = __float2half_rn(v);
    if (__half2float(h) != v) ++bad;
    y16[i] = h;
  }
  if (__syncthreads_or(bad)) {
    if (bad) atomicAdd(inexact, bad);
  }
}

// One pass over the spike counts for everything an E-step needs from them (reference decoder.py:40: the
// gammaln(y+1) term depends on y only): fp16 copy [T, ld16] (+ optional column of ones at index N, zero padding),
// exactness flag, lgam[t] = sum_n m_n lgamma(y[t,n]+1) and optionally ysum[t] = sum_n m_n y[t,n].
// One warp per time bin; VEC: rows are 16-byte aligned and N % 4 == 0 (float4 loads, 8-byte stores).
__device__ __forceinline__ float lgamma1p_count(float v) {
  // log(n!) for the small integer counts that make up spike data; anything else through lgammaf
  if (v == 0.f || v == 1.f) return 0.f;
  if (v == 2.f) return 0.69314718055994531f;
  if (v == 3.f) return 1.7917594692280550f;
  if (v == 4.f) return 3.1780538303479458f;
  if (v == 5.f) return 4.7874917427820458f;
  if (v == 6.f) return 6.5792512120101012f;
  return lgammaf(v + 1.f);
}

template <bool VEC>
__global__ void __launch_bounds__(256)
counts_prepare_kernel(int64_t T, int N, const float* __restrict__ y, int64_t ldy, const float* __restrict__ ma,
                      __half* __restrict__ y16, int64_t ld16, int ones_col, int* __restrict__ inexact,
                      float* __restrict__ lgam, float* __restrict__ ysum) {
  const int lane = threadIdx.x & 31;
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const float* row = y + (size_t)t * ldy;
  __half* orow = y16 + (size_t)t * ld16;
  float acc = 0.f, ys = 0.f;
  int bad = 0;
  if (VEC) {
    const int n4 = N >> 2;
    for (int j0 = 0; j0 < n4; j0 += 128) {         // four independent 16-byte loads per lane in flight
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * 32 + lane;
        v[u] = j < n4 ? __ldcs(reinterpret_cast<const float4*>(row) + j) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = j0 + u * 32 + lane;
        if (j >= n4) continue;
        const float x[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        float m[4] = {1.f, 1.f, 1.f, 1.f};
        if (ma) {
          const float4 m4 = __ldg(reinterpret_cast<const float4*>(ma) + j);
          m[0] = m4.x; m[1] = m4.y; m[2] = m4.z; m[3] = m4.w;
        }
        __half h[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          h[e] = __float2half_rn(x[e]);
          bad |= (__half2float(h[e]) != x[e]);
          acc = fmaf(m[e], lgamma1p_count(x[e]), acc);
          ys = fmaf(m[e], x[e], ys);
        }
        uint2 pk;
        pk.x = (uint32_t)__half_as_ushort(h[0]) | ((uint32_t)__half_as_ushort(h[1]) << 16);
        pk.y = (uint32_t)__half_as_ushort(h[2]) | ((uint32_t)__half_as_ushort(h[3]) << 16);
        reinterpret_cast<uint2*>(orow)[j] = pk;
      }
    }
  } else {
    for (int n = lane; n < N; n += 32) {
      const float x = row[n];
      const float m = ma ? ma[n] : 1.f;
      const __half h = __float2half_rn(x);
      bad |= (__half2float(h) != x);
      acc = fmaf(m, lgamma1p_count(x), acc);
      ys = fmaf(m, x, ys);
      orow[n] = h;
    }
  }
  for (int n = N + lane; n < (int)ld16; n += 32)
    orow[n] = (ones_col && n == N) ? __float2half_rn(1.f) : __float2half_rn(0.f);
  acc = warp_sum(acc);
  ys = warp_sum(ys);
  if (lane == 0) {
    lgam[t] = acc;
    if (ysum) ysum[t] = ys;
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicAdd(inexact, 1);
}

// Circularly shifted counts of a shuffle test (np.roll per neuron, reference test.py:22-23), n_shift shuffles stacked
// along time: y16[b*T + t, n] = yT[n, (t - shifts[b*N + n]) mod T] and lgam[b*T + t] = sum_n m_n lgamma(.+1).
// The source is neuron-major, so a neuron's shifted window of SH_TT bins is one contiguous (once wrapped) run: a CTA
// copies the windows of a slab of SH_NS neurons into a time-major shared tile (coalesced along t), then every warp
// emits SH_TT / 8 rows of it.  lgam reproduces counts_prepare_kernel bit for bit: lane l sums the neurons n with
// (n >> 2) % 32 == l (VEC, float4 groups) or n % 32 == l, in increasing n, with the same fmaf and the same
// warp_sum.  SH_NS is a multiple of 128, so that per-lane order survives the slab loop.
constexpr int SH_TT = 64;                 // output bins per CTA
constexpr int SH_NS = 256;                // neurons per shared-memory slab
constexpr int SH_STR = SH_NS + 2;         // tile row stride (halves): 129 words, odd -> conflict-free transpose
constexpr int SH_THREADS = 256;
constexpr int SH_RPW = SH_TT / (SH_THREADS / 32);   // rows per warp

template <bool VEC>
__global__ void __launch_bounds__(SH_THREADS)
counts_prepare_shifted_kernel(int64_t T, int N, int64_t n_tiles, const __half* __restrict__ yT, int64_t ld_src,
                              const int* __restrict__ shifts, const float* __restrict__ ma, __half* __restrict__ y16,
                              int64_t ld16, float* __restrict__ lgam) {
  __shared__ __align__(16) __half tile[SH_TT * SH_STR];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t b = blockIdx.x / n_tiles;
  const int64_t t0 = (blockIdx.x - b * n_tiles) * SH_TT;
  const int* sh = shifts + b * N;
  float acc[SH_RPW];
#pragma unroll
  for (int r = 0; r < SH_RPW; ++r) acc[r] = 0.f;
  for (int n0 = 0; n0 < N; n0 += SH_NS) {
    const int ns = min(SH_NS, N - n0);
    if (n0) __syncthreads();                      // previous slab fully emitted
    // load: consecutive threads take consecutive bins of one neuron
    for (int i = threadIdx.x; i < ns * SH_TT; i += SH_THREADS) {
      const int nl = i / SH_TT, tt = i - nl * SH_TT;
      const int64_t t = t0 + tt;
      __half h = __ushort_as_half(0);
      if (t < T) {
        int64_t src = t - sh[n0 + nl];
        if (src < 0) src += T;
        h = yT[(size_t)(n0 + nl) * ld_src + src];
      }
      tile[tt * SH_STR + nl] = h;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < SH_RPW; ++r) {
      const int tt = warp * SH_RPW + r;
      const int64_t t = t0 + tt;
      if (t >= T) break;
      const __half* trow = tile + tt * SH_STR;
      __half* orow = y16 + (size_t)(b * T + t) * ld16 + n0;
      if (VEC) {
        for (int jl = lane; jl < (ns >> 2); jl += 32) {
          const __half2 p0 = *reinterpret_cast<const __half2*>(trow + 4 * jl);
          const __half2 p1 = *reinterpret_cast<const __half2*>(trow + 4 * jl + 2);
          const float x[4] = {__low2float(p0), __high2float(p0), __low2float(p1), __high2float(p1)};
          float m[4] = {1.f, 1.f, 1.f, 1.f};
          if (ma) {
            const float4 m4 = __ldg(reinterpret_cast<const float4*>(ma + n0) + jl);
            m[0] = m4.x; m[1] = m4.y; m[2] = m4.z; m[3] = m4.w;
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) acc[r] = fmaf(m[e], lgamma1p_count(x[e]), acc[r]);
          uint2 pk;
          pk.x = *reinterpret_cast<const uint32_t*>(&p0);
          pk.y = *reinterpret_cast<const uint32_t*>(&p1);
          reinterpret_cast<uint2*>(orow)[jl] = pk;
        }
      } else {
        for (int nl = lane; nl < ns; nl += 32) {
          const __half h = trow[nl];
          const float m = ma ? ma[n0 + nl] : 1.f;
          acc[r] = fmaf(m, lgamma1p_count(__half2float(h)), acc[r]);
          orow[nl] = h;
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < SH_RPW; ++r) {
    const int64_t t = t0 + warp * SH_RPW + r;
    if (t >= T) break;
    __half* orow = y16 + (size_t)(b * T + t) * ld16;
    for (int n = N + lane; n < (int)ld16; n += 32) orow[n] = __ushort_as_half(0);
    const float s = warp_sum(acc[r]);
    if (lane == 0) lgam[b * T + t] = s;
  }
}

// loglam pieces [2][Kpad][ld16]; rows >= K and columns >= N are zero.  One CTA per padded row.
__global__ void emission_prepare_f16_kernel(int K, int N, const float* __restrict__ tuning,
                                            const float* __restrict__ ma_neuron, float dt, int Kpad, int64_t ld16,
                                            __half* __restrict__ L16, float* __restrict__ lam_sum) {
  const int k = blockIdx.x;
  __half* hi = L16 + (size_t)k * ld16;
  __half* lo = L16 + ((size_t)Kpad + k) * ld16;
  double acc = 0.0;
  for (int n = threadIdx.x; n < (int)ld16; n += blockDim.x) {
    float v = 0.f;
    if (k < K && n < N) {
      const float m = ma_neuron ? ma_neuron[n] : 1.f;
      const float lam = tuning[(size_t)k * N + n] * dt + kLamFloor;
      v = m * logf(lam);
      acc += (double)(m * lam);
    }
    const __half h = __float2half_rn(v);
    hi[n] = h;
    lo[n] = __float2half_rn(v - __half2float(h));
  }
  if (k >= K) return;
  acc = warp_sum_d(acc);
  __shared__ double sm[32];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sm[w];
    lam_sum[k] = (float)s;
  }
}

// ---------------------------------------------------------------------------------------------
// emission: K-major operands
// ---------------------------------------------------------------------------------------------
struct EmissionTcParams {
  int64_t T;
  int K, Kpad, BN, n_kblocks, n_mtiles, n_ntiles, stages, stagger, ep_nbuf;
  uint32_t idesc, tmem_cols;
  const float* lam_sum;
  const float* lgam;
  const float* ma_latent;
  float* ll;
  int64_t ldll;
};

constexpr int EM_PB = 2;   // fp16 pieces of loglam
constexpr int EM_MI = 2;   // 128-row tiles per work unit: both share every right-hand tile fetched from L2
constexpr int EP_BUF_BYTES = 4096;   // epilogue staging tile: 32 rows x 128 B
constexpr int EM_THREADS = 384;      // warps: 0 TMA producer, 1 MMA issuer, 2 TMEM allocator, 4-7 / 8-11 epilogue

__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ void sts_f4(uint32_t saddr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
}

// Work unit = 256 time bins x BN latent bins: two TMEM accumulators side by side, one pass over the neurons.
// The main loop is bound by the L2 -> shared-memory feed of the (small, shared) right-hand operand, so a unit
// uses each right-hand tile for two row tiles.  Epilogue: one set of four warps per accumulator; every warp
// drains its 32 TMEM lanes in chunks of 32 columns -> registers (next chunk's load in flight) -> swizzled
// staging tile -> TMA store (full 128-byte lines; rows past T and columns past K are clipped by the tensor
// map).  An accumulator is handed back to the MMA warp as soon as its last chunk is in registers, and the MMA
// warp starts a unit with the accumulator-0 products of the first two K blocks, so the stores and most of the
// drain run under the next unit's MMAs.
__global__ void __launch_bounds__(EM_THREADS, 1)
emission_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const __grid_constant__ CUtensorMap tmC32, const __grid_constant__ CUtensorMap tmC16,
                   const EmissionTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = p.BN;
  const uint32_t b_bytes = (uint32_t)BN * TC_BK * 2;
  const uint32_t stage_bytes = EM_MI * TC_A_BYTES + EM_PB * b_bytes;
  uint8_t* stg_base = smem + (size_t)p.stages * stage_bytes;                      // 1024-aligned
  float* ls_s = reinterpret_cast<float*>(stg_base + (size_t)8 * p.ep_nbuf * EP_BUF_BYTES);   // [Kpad]
  uint64_t* full = reinterpret_cast<uint64_t*>(ls_s + ((p.Kpad + 3) & ~3));
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + EM_MI);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    for (int b = 0; b < EM_MI; ++b) mbar_init(&tempty[b], 128);
    fence_barrier_init();
  }
  // per-column term of the epilogue: sum_n lam (NaN marks a masked-out latent bin)
  for (int k = threadIdx.x; k < p.Kpad; k += blockDim.x) {
    float v = 0.f;
    if (k < p.K) {
      v = p.lam_sum[k];
      if (p.ma_latent && p.ma_latent[k] == 0.f) v = __int_as_float(0x7fc00000);
    }
    ls_s[k] = v;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); tma_prefetch_desc(&tmC32); tma_prefetch_desc(&tmC16);
  }
  if (warp == 2) { tmem_alloc(tmem_slot, p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_mpairs = (p.n_mtiles + EM_MI - 1) / EM_MI;
  const int n_units = n_mpairs * p.n_ntiles;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      // experiment knob (p.stagger): every CTA walks the K blocks in a different rotation; off by default because
      // it makes the fp32 accumulation order, hence the low bits of ll, depend on the tile's position
      const int kb0 = p.stagger ? (int)(blockIdx.x % p.n_kblocks) : 0;
      for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
        const int mp = unit / p.n_ntiles, nt = unit % p.n_ntiles;
        for (int kb = 0; kb < p.n_kblocks; ++kb) {
          int kbe = kb + kb0;
          if (kbe >= p.n_kblocks) kbe -= p.n_kblocks;
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + (size_t)stage * stage_bytes;
          mbar_arrive_expect_tx(&full[stage], stage_bytes);
#pragma unroll
          for (int mi = 0; mi < EM_MI; ++mi)      // rows past T are zero-filled by the TMA unit
            tma_load_2d(sA + mi * TC_A_BYTES, &tmA, &full[stage], kbe * TC_BK, (mp * EM_MI + mi) * TC_BM);
#pragma unroll
          for (int pc = 0; pc < EM_PB; ++pc)
            tma_load_2d(sA + EM_MI * TC_A_BYTES + pc * b_bytes, &tmB, &full[stage], kbe * TC_BK,
                        pc * p.Kpad + nt * BN);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;
      // all MMAs of K block `first` (first = this accumulator has nothing accumulated yet) for row tile mi
      auto issue = [&](int st, int mi, bool first) {
        const uint32_t sA = smem_u32(smem + (size_t)st * stage_bytes);
        const uint32_t d_tmem = tmem_base + (uint32_t)(mi * BN);
#pragma unroll
        for (int pc = 0; pc < EM_PB; ++pc) {
          const uint32_t sB = sA + EM_MI * TC_A_BYTES + pc * b_bytes;
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            const uint64_t ad = make_smem_desc(sA + mi * TC_A_BYTES + k * 32, 16, 1024);
            const uint64_t bd = make_smem_desc(sB + k * 32, 16, 1024);
            mma_f16_ss(d_tmem, ad, bd, p.idesc, (first && pc == 0 && k == 0) ? 0u : 1u);
          }
        }
      };
      for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
        const uint32_t drained = (uint32_t)(it & 1) ^ 1;      // parity of "the previous unit's epilogue is done"
        int kb = 0;
        if (p.n_kblocks >= 2 && p.stages >= 2) {
          // accumulator 0 is drained first: run its products of the first two K blocks while accumulator 1 drains
          const int s0 = stage; const uint32_t ph0 = phase;
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
          const int s1 = stage; const uint32_t ph1 = phase;
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
          mbar_wait(&full[s0], ph0);
          mbar_wait(&tempty[0], drained);
          tc_fence_after();
          issue(s0, 0, true);
          mbar_wait(&full[s1], ph1);
          tc_fence_after();
          issue(s1, 0, false);
          mbar_wait(&tempty[1], drained);
          tc_fence_after();
          issue(s0, 1, true);
          mma_commit(&empty[s0]);
          issue(s1, 1, false);
          mma_commit(&empty[s1]);
          kb = 2;
        }
        for (; kb < p.n_kblocks; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
#pragma unroll
          for (int mi = 0; mi < EM_MI; ++mi) {
            if (kb == 0) {
              mbar_wait(&tempty[mi], drained);
              tc_fence_after();
            }
            issue(stage, mi, kb == 0);
          }
          mma_commit(&empty[stage]);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        mma_commit(tfull);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int mi = (warp - 4) >> 2;              // accumulator (row tile) this warp set drains
    const uint32_t stg = smem_u32(stg_base + (size_t)(warp - 4) * p.ep_nbuf * EP_BUF_BYTES);
    const uint32_t ls_addr = smem_u32(ls_s);
    const uint32_t stg_row128 = (uint32_t)lane * 128u, sw128 = (uint32_t)(lane & 7);
    const uint32_t stg_row64 = (uint32_t)lane * 64u, sw64 = (uint32_t)((lane >> 1) & 3);
    const int nch = (BN + 31) / 32;              // chunks per accumulator (BN is a multiple of 16: the last may be 16 wide)
    const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mi * BN);
    const bool masked = p.ma_latent != nullptr;
    int it = 0, buf = 0;
    for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x, ++it) {
      const int mp = unit / p.n_ntiles, nt = unit % p.n_ntiles;
      const int64_t t0 = (int64_t)(mp * EM_MI + mi) * TC_BM + q * 32;     // first row of this warp
      const float lg = (t0 + lane) < p.T ? __ldg(p.lgam + t0 + lane) : 0.f;
      const bool rows_ok = t0 < p.T;
      mbar_wait(tfull, (uint32_t)(it & 1));
      tc_fence_after();

      auto issue = [&](int c, uint32_t (&r)[32]) {
        const int c0 = c * 32;
        if (c0 + 32 <= BN) tmem_ld_x32(tbase + (uint32_t)c0, r); else tmem_ld_x16_of32(tbase + (uint32_t)c0, r);
      };
      auto process = [&](int c, uint32_t (&r)[32]) {
        const int c0 = c * 32;
        if (c == nch - 1) {                      // the last chunk of this accumulator has left TMEM
          tc_fence_before();
          mbar_arrive(&tempty[mi]);
        }
        const bool wide = c0 + 32 <= BN;
        // the staging tile about to be overwritten must have been read by its TMA store
        if (lane == 0) {
          // at most ep_nbuf - 1 earlier stores may still be reading their staging tiles
          if (p.ep_nbuf == 1) bulk_wait_read<0>(); else if (p.ep_nbuf == 2) bulk_wait_read<1>(); else bulk_wait_read<2>();
        }
        __syncwarp();
        const uint32_t sb = stg + (uint32_t)buf * EP_BUF_BYTES;
        const uint32_t lsp = ls_addr + (uint32_t)(nt * BN + c0) * 4u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (!wide && j >= 4) break;
          const float4 l4 = lds_f4(lsp + 16u * j);
          float4 v;
          v.x = __uint_as_float(r[4 * j + 0]) - l4.x - lg;
          v.y = __uint_as_float(r[4 * j + 1]) - l4.y - lg;
          v.z = __uint_as_float(r[4 * j + 2]) - l4.z - lg;
          v.w = __uint_as_float(r[4 * j + 3]) - l4.w - lg;
          if (masked) {
            if (l4.x != l4.x) v.x = kVeryNegLL;
            if (l4.y != l4.y) v.y = kVeryNegLL;
            if (l4.z != l4.z) v.z = kVeryNegLL;
            if (l4.w != l4.w) v.w = kVeryNegLL;
          }
          const uint32_t off = wide ? stg_row128 + (((uint32_t)j ^ sw128) << 4)
                                    : stg_row64 + (((uint32_t)j ^ sw64) << 4);
          sts_f4(sb + off, v);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          const int col0 = nt * BN + c0;
          if (rows_ok && col0 < p.K) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(reinterpret_cast<uint64_t>(wide ? &tmC32 : &tmC16)), "r"(sb), "r"(col0), "r"((int)t0)
                         : "memory");
          }
          bulk_commit();
        }
        if (++buf == p.ep_nbuf) buf = 0;
      };

      uint32_t ra[32], rb[32];
      issue(0, ra);
      for (int c = 0; c < nch; c += 2) {
        tmem_ld_wait();
        if (c + 1 < nch) issue(c + 1, rb);
        process(c, ra);
        if (c + 1 < nch) {
          tmem_ld_wait();
          if (c + 2 < nch) issue(c + 2, ra);
          process(c + 1, rb);
        }
      }
    }
    if (lane == 0) bulk_wait_read<0>();          // shared memory must outlive the last stores' reads
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, p.tmem_cols); }
}

// CTA-pair version (cta_group::2).  The single-CTA kernel above is bound by the L2 -> shared-memory feed: per K
// block it pulls 32 KB of counts and 52 KB of log-rate pieces for 256 x 208 outputs.  Here two CTAs of a cluster
// (the two SMs of a TPC) share every right-hand tile: a work unit is 512 time bins x BN latent bins, each CTA
// loads its own 2 x 128 rows of counts and HALF of the log-rate rows (58 KB per CTA and K block instead of 84),
// and the leader issues MMAs of M = 256 that read both halves; each CTA accumulates and drains its own 128-lane
// accumulators.  Barriers: both CTAs' loads count on the leader's `full`; the leader's commits arrive on both
// CTAs' `empty` / `tfull` (multicast); both CTAs' epilogue warps arrive on the leader's `tempty`.
__global__ void __launch_bounds__(EM_THREADS, 1)
emission_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh,
                    const __grid_constant__ CUtensorMap tmC32, const __grid_constant__ CUtensorMap tmC16,
                    const EmissionTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = p.BN;
  const uint32_t bh_bytes = (uint32_t)(BN / 2) * TC_BK * 2;          // this CTA's half of one log-rate piece
  const uint32_t stage_bytes = EM_MI * TC_A_BYTES + EM_PB * bh_bytes;
  uint8_t* stg_base = smem + (size_t)p.stages * stage_bytes;                      // 1024-aligned
  float* ls_s = reinterpret_cast<float*>(stg_base + (size_t)8 * p.ep_nbuf * EP_BUF_BYTES);   // [Kpad]
  uint64_t* full = reinterpret_cast<uint64_t*>(ls_s + ((p.Kpad + 3) & ~3));
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + EM_MI);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();               // 0 = leader
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    for (int b = 0; b < EM_MI; ++b) mbar_init(&tempty[b], 256);     // 128 epilogue threads of each CTA
    fence_barrier_init();
  }
  for (int k = threadIdx.x; k < p.Kpad; k += blockDim.x) {
    float v = 0.f;
    if (k < p.K) {
      v = p.lam_sum[k];
      if (p.ma_latent && p.ma_latent[k] == 0.f) v = __int_as_float(0x7fc00000);
    }
    ls_s[k] = v;
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmBh); tma_prefetch_desc(&tmC32); tma_prefetch_desc(&tmC16);
  }
  if (warp == 2) { tmem_alloc2(tmem_slot, p.tmem_cols); tmem_relinquish2(); }
  tc_fence_before();
  cluster_sync_all();                                    // barriers and TMEM of BOTH CTAs are ready
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_mquads = (p.n_mtiles + 2 * EM_MI - 1) / (2 * EM_MI);          // 512-row groups
  const int n_units = n_mquads * p.n_ntiles;
  const int cluster = blockIdx.x >> 1, n_clusters = gridDim.x >> 1;
  // row tile of accumulator mi of this CTA inside the 512-row group: MMA mi covers tiles (2 mi, 2 mi + 1)
  auto row_tile = [&](int mq, int mi) { return mq * (2 * EM_MI) + 2 * mi + (int)rank; };

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int unit = cluster; unit < n_units; unit += n_clusters) {
        const int mq = unit / p.n_ntiles, nt = unit % p.n_ntiles;
        for (int kb = 0; kb < p.n_kblocks; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + (size_t)stage * stage_bytes;
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * stage_bytes);     // both CTAs' bytes
#pragma unroll
          for (int mi = 0; mi < EM_MI; ++mi)      // rows past T are zero-filled by the TMA unit
            tma_load_2d_pair(sA + mi * TC_A_BYTES, &tmA, &full[stage], kb * TC_BK, row_tile(mq, mi) * TC_BM);
#pragma unroll
          for (int pc = 0; pc < EM_PB; ++pc)
            tma_load_2d_pair(sA + EM_MI * TC_A_BYTES + pc * bh_bytes, &tmBh, &full[stage], kb * TC_BK,
                             pc * p.Kpad + nt * BN + (int)rank * (BN / 2));
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;
      auto issue = [&](int st, int mi, bool first) {
        const uint32_t sA = smem_u32(smem + (size_t)st * stage_bytes);
        const uint32_t d_tmem = tmem_base + (uint32_t)(mi * BN);
#pragma unroll
        for (int pc = 0; pc < EM_PB; ++pc) {
          const uint32_t sB = sA + EM_MI * TC_A_BYTES + pc * bh_bytes;
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            const uint64_t ad = make_smem_desc(sA + mi * TC_A_BYTES + k * 32, 16, 1024);
            const uint64_t bd = make_smem_desc(sB + k * 32, 16, 1024);
            mma_f16_ss2(d_tmem, ad, bd, p.idesc, (first && pc == 0 && k == 0) ? 0u : 1u);
          }
        }
      };
      for (int unit = cluster; unit < n_units; unit += n_clusters, ++it) {
        const uint32_t drained = (uint32_t)(it & 1) ^ 1;      // parity of "the previous unit's epilogues are done"
        int kb = 0;
        if (p.n_kblocks >= 2 && p.stages >= 2) {
          const int s0 = stage; const uint32_t ph0 = phase;
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
          const int s1 = stage; const uint32_t ph1 = phase;
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
          mbar_wait(&full[s0], ph0);
          mbar_wait(&tempty[0], drained);
          tc_fence_after();
          issue(s0, 0, true);
          mbar_wait(&full[s1], ph1);
          tc_fence_after();
          issue(s1, 0, false);
          mbar_wait(&tempty[1], drained);
          tc_fence_after();
          issue(s0, 1, true);
          mma_commit2(&empty[s0], 3);
          issue(s1, 1, false);
          mma_commit2(&empty[s1], 3);
          kb = 2;
        }
        for (; kb < p.n_kblocks; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
#pragma unroll
          for (int mi = 0; mi < EM_MI; ++mi) {
            if (kb == 0) {
              mbar_wait(&tempty[mi], drained);
              tc_fence_after();
            }
            issue(stage, mi, kb == 0);
          }
          mma_commit2(&empty[stage], 3);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        mma_commit2(tfull, 3);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    const int mi = (warp - 4) >> 2;              // accumulator (row tile) this warp set drains
    const uint32_t stg = smem_u32(stg_base + (size_t)(warp - 4) * p.ep_nbuf * EP_BUF_BYTES);
    const uint32_t ls_addr = smem_u32(ls_s);
    const uint32_t stg_row128 = (uint32_t)lane * 128u, sw128 = (uint32_t)(lane & 7);
    const uint32_t stg_row64 = (uint32_t)lane * 64u, sw64 = (uint32_t)((lane >> 1) & 3);
    const int nch = (BN + 31) / 32;
    const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mi * BN);
    const bool masked = p.ma_latent != nullptr;
    int it = 0, buf = 0;
    for (int unit = cluster; unit < n_units; unit += n_clusters, ++it) {
      const int mq = unit / p.n_ntiles, nt = unit % p.n_ntiles;
      const int64_t t0 = (int64_t)row_tile(mq, mi) * TC_BM + q * 32;     // first row of this warp
      const float lg = (t0 + lane) < p.T ? __ldg(p.lgam + t0 + lane) : 0.f;
      const bool rows_ok = t0 < p.T;
      mbar_wait(tfull, (uint32_t)(it & 1));
      tc_fence_after();

      auto issue = [&](int c, uint32_t (&r)[32]) {
        const int c0 = c * 32;
        if (c0 + 32 <= BN) tmem_ld_x32(tbase + (uint32_t)c0, r); else tmem_ld_x16_of32(tbase + (uint32_t)c0, r);
      };
      auto process = [&](int c, uint32_t (&r)[32]) {
        const int c0 = c * 32;
        if (c == nch - 1) {                      // the last chunk of this accumulator has left TMEM
          tc_fence_before();
          if (rank == 0) mbar_arrive(&tempty[mi]); else mbar_arrive_cluster(&tempty[mi], 0);
        }
        const bool wide = c0 + 32 <= BN;
        if (lane == 0) {
          // at most ep_nbuf - 1 earlier stores may still be reading their staging tiles
          if (p.ep_nbuf == 1) bulk_wait_read<0>(); else if (p.ep_nbuf == 2) bulk_wait_read<1>(); else bulk_wait_read<2>();
        }
        __syncwarp();
        const uint32_t sb = stg + (uint32_t)buf * EP_BUF_BYTES;
        const uint32_t lsp = ls_addr + (uint32_t)(nt * BN + c0) * 4u;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (!wide && j >= 4) break;
          const float4 l4 = lds_f4(lsp + 16u * j);
          float4 v;
          v.x = __uint_as_float(r[4 * j + 0]) - l4.x - lg;
          v.y = __uint_as_float(r[4 * j + 1]) - l4.y - lg;
          v.z = __uint_as_float(r[4 * j + 2]) - l4.z - lg;
          v.w = __uint_as_float(r[4 * j + 3]) - l4.w - lg;
          if (masked) {
            if (l4.x != l4.x) v.x = kVeryNegLL;
            if (l4.y != l4.y) v.y = kVeryNegLL;
            if (l4.z != l4.z) v.z = kVeryNegLL;
            if (l4.w != l4.w) v.w = kVeryNegLL;
          }
          const uint32_t off = wide ? stg_row128 + (((uint32_t)j ^ sw128) << 4)
                                    : stg_row64 + (((uint32_t)j ^ sw64) << 4);
          sts_f4(sb + off, v);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          const int col0 = nt * BN + c0;
          if (rows_ok && col0 < p.K) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                         ::"l"(reinterpret_cast<uint64_t>(wide ? &tmC32 : &tmC16)), "r"(sb), "r"(col0), "r"((int)t0)
                         : "memory");
          }
          bulk_commit();
        }
        if (++buf == p.ep_nbuf) buf = 0;
      };

      uint32_t ra[32], rb[32];
      issue(0, ra);
      for (int c = 0; c < nch; c += 2) {
        tmem_ld_wait();
        if (c + 1 < nch) issue(c + 1, rb);
        process(c, ra);
        if (c + 1 < nch) {
          tmem_ld_wait();
          if (c + 2 < nch) issue(c + 2, ra);
          process(c + 1, rb);
        }
      }
    }
    if (lane == 0) bulk_wait_read<0>();          // shared memory must outlive the last stores' reads
  }
  tc_fence_before();
  cluster_sync_all();                            // the peer may still read this CTA's shared memory / arrive here
  if (warp == 2) { tc_fence_after(); tmem_dealloc2(tmem_base, p.tmem_cols); }
}

// previous structure (one 128-row tile per unit, double-buffered accumulator), kept selectable for experiments
__global__ void __launch_bounds__(TC_THREADS, 1)
emission_tc_kernel_v1(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                   const EmissionTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int BN = p.BN;
  const uint32_t b_bytes = (uint32_t)BN * TC_BK * 2;
  const uint32_t stage_bytes = TC_A_BYTES + EM_PB * b_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 128); }
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB); }
  if (warp == 2) { tmem_alloc(tmem_slot, p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_tiles = p.n_mtiles * p.n_ntiles;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int mt = tile / p.n_ntiles, nt = tile % p.n_ntiles;
        const int kb0 = p.stagger ? (int)(blockIdx.x % p.n_kblocks) : 0;
        for (int kb = 0; kb < p.n_kblocks; ++kb) {
          int kbe = kb + kb0;
          if (kbe >= p.n_kblocks) kbe -= p.n_kblocks;
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + (size_t)stage * stage_bytes;
          mbar_arrive_expect_tx(&full[stage], stage_bytes);
          tma_load_2d(sA, &tmA, &full[stage], kbe * TC_BK, mt * TC_BM);
#pragma unroll
          for (int pc = 0; pc < EM_PB; ++pc)
            tma_load_2d(sA + TC_A_BYTES + pc * b_bytes, &tmB, &full[stage], kbe * TC_BK, pc * p.Kpad + nt * BN);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0; int it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&tempty[buf], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * BN);
        for (int kb = 0; kb < p.n_kblocks; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sA = smem_u32(smem + (size_t)stage * stage_bytes);
#pragma unroll
          for (int pc = 0; pc < EM_PB; ++pc) {
            const uint32_t sB = sA + TC_A_BYTES + pc * b_bytes;
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k) {
              const uint64_t ad = make_smem_desc(sA + k * 32, 16, 1024);
              const uint64_t bd = make_smem_desc(sB + k * 32, 16, 1024);
              mma_f16_ss(d_tmem, ad, bd, p.idesc, (kb | pc | k) != 0);
            }
          }
          mma_commit(&empty[stage]);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        mma_commit(&tfull[buf]);
      }
    }
  } else if (warp >= 4) {
    const int q = warp & 3;                      // TMEM lane quarter this warp may access
    int it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
      const int mt = tile / p.n_ntiles, nt = tile % p.n_ntiles;
      const int buf = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tfull[buf], acc_phase);
      tc_fence_after();
      const int64_t t = (int64_t)mt * TC_BM + q * 32 + lane;
      const bool t_ok = t < p.T;
      const float lg = t_ok ? p.lgam[t] : 0.f;
      float* orow = p.ll + (size_t)(t_ok ? t : 0) * p.ldll;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN);
      const bool vec_ok = (p.ldll & 3) == 0;
      for (int c0 = 0; c0 < BN; c0 += 16) {
        uint32_t r[16];
        tmem_ld_x16(taddr + c0, r);
        tmem_ld_wait();
        const int k0 = nt * BN + c0;
        if (t_ok && k0 < p.K) {
          float v[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int k = k0 + j;
            float x = __uint_as_float(r[j]);
            if (k < p.K) {
              x = x - __ldg(p.lam_sum + k) - lg;
              if (p.ma_latent && __ldg(p.ma_latent + k) == 0.f) x = kVeryNegLL;
            }
            v[j] = x;
          }
          if (vec_ok && k0 + 16 <= p.K) {
#pragma unroll
            for (int j = 0; j < 16; j += 4)
              *reinterpret_cast<float4*>(orow + k0 + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (k0 + j < p.K) orow[k0 + j] = v[j];
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty[buf]);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, p.tmem_cols); }
}

static uint32_t pow2_cols(int c) {
  uint32_t v = 32;
  while ((int)v < c) v <<= 1;
  return v;
}

}  // namespace pmg

// BN = accumulator columns per tile: K split into ceil(K/256) tiles, rounded up to 16
extern "C" int pmg_emission_tile_n(int K) {
  if (K <= 0) return 0;
  const int nt = (K + 255) / 256;
  int bn = (K + nt - 1) / nt;
  bn = (bn + 15) / 16 * 16;
  return bn;
}

extern "C" int pmg_counts_to_f16(int64_t T, int N, const float* y, int64_t ldy, void* y16, int64_t ld16,
                                 int* inexact_count, pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || !y || !y16 || !inexact_count || ldy < N || ld16 < N || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  PMG_CUDA_CHECK(cudaMemsetAsync(inexact_count, 0, sizeof(int), st));
  pmg::counts_to_f16_kernel<<<148 * 8, 256, 0, st>>>(T, N, y, ldy, (__half*)y16, ld16, inexact_count);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_counts_prepare(int64_t T, int N, const float* y, int64_t ldy, const float* ma_neuron, void* y16,
                                  int64_t ld16, int ones_col, int* inexact_count, float* lgam, float* ysum,
                                  pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || !y || !y16 || !inexact_count || !lgam || ldy < N || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  if (ld16 < N + (ones_col ? 1 : 0)) return PMG_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  PMG_CUDA_CHECK(cudaMemsetAsync(inexact_count, 0, sizeof(int), st));
  const bool vec = (N & 3) == 0 && (ldy & 3) == 0 && ((uintptr_t)y & 15) == 0 && (!ma_neuron || ((uintptr_t)ma_neuron & 15) == 0);
  const unsigned grid = (unsigned)pmg::cdiv(T, 8);
  if (vec)
    pmg::counts_prepare_kernel<true><<<grid, 256, 0, st>>>(T, N, y, ldy, ma_neuron, (__half*)y16, ld16, ones_col,
                                                           inexact_count, lgam, ysum);
  else
    pmg::counts_prepare_kernel<false><<<grid, 256, 0, st>>>(T, N, y, ldy, ma_neuron, (__half*)y16, ld16, ones_col,
                                                            inexact_count, lgam, ysum);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_counts_prepare_shifted(int64_t T, int N, int n_shift, const void* yT16, int64_t ld_src,
                                          const int* shifts, const float* ma_neuron, void* y16, int64_t ld16,
                                          float* lgam, pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || n_shift <= 0 || !yT16 || !shifts || !y16 || !lgam) return PMG_ERR_BAD_ARG;
  if (ld_src < T || ld16 < N || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  if ((uintptr_t)y16 & 15) return PMG_ERR_ALIGNMENT;
  const int64_t n_tiles = (T + pmg::SH_TT - 1) / pmg::SH_TT;
  if (n_tiles * n_shift > 0x7fffffffLL) return PMG_ERR_UNSUPPORTED_SHAPE;
  // same float4 / scalar choice as pmg_counts_prepare on a contiguous [T, N] matrix (the lane order of lgam)
  const bool vec = (N & 3) == 0 && (!ma_neuron || ((uintptr_t)ma_neuron & 15) == 0);
  const unsigned grid = (unsigned)(n_tiles * n_shift);
  cudaStream_t st = (cudaStream_t)stream;
  if (vec)
    pmg::counts_prepare_shifted_kernel<true><<<grid, pmg::SH_THREADS, 0, st>>>(
        T, N, n_tiles, (const __half*)yT16, ld_src, shifts, ma_neuron, (__half*)y16, ld16, lgam);
  else
    pmg::counts_prepare_shifted_kernel<false><<<grid, pmg::SH_THREADS, 0, st>>>(
        T, N, n_tiles, (const __half*)yT16, ld_src, shifts, ma_neuron, (__half*)y16, ld16, lgam);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_prepare_f16(int K, int N, const float* tuning, const float* ma_neuron, float dt,
                                        int Kpad, int64_t ld16, void* loglam16, float* lam_sum,
                                        pmg_stream_t stream) {
  if (K <= 0 || N <= 0 || !tuning || !loglam16 || !lam_sum || Kpad < K || ld16 < N || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  pmg::emission_prepare_f16_kernel<<<Kpad, 128, 0, (cudaStream_t)stream>>>(K, N, tuning, ma_neuron, dt, Kpad, ld16,
                                                                          (__half*)loglam16, lam_sum);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_poisson_f16(int64_t T, int N, int K, const void* y16, int64_t ld16,
                                        const void* loglam16, int Kpad, const float* lam_sum, const float* lgam,
                                        const float* ma_latent, float* ll, int64_t ldll, pmg_stream_t stream) {
  using namespace pmg;
  if (T <= 0 || N <= 0 || K <= 0 || !y16 || !loglam16 || !lam_sum || !lgam || !ll) return PMG_ERR_BAD_ARG;
  if (ld16 < N || (ld16 & 7) || ldll < K) return PMG_ERR_BAD_ARG;
  if (((uintptr_t)y16 & 15) || ((uintptr_t)loglam16 & 15)) return PMG_ERR_ALIGNMENT;
  const int BN = pmg_emission_tile_n(K);
  const int n_ntiles = (K + BN - 1) / BN;
  if (Kpad != n_ntiles * BN) return PMG_ERR_BAD_ARG;
  if (T > ((int64_t)1 << 31) - 256) return PMG_ERR_UNSUPPORTED_SHAPE;

  CUtensorMap tmA, tmB;
  int rc = make_tmap_f16(&tmA, y16, (uint64_t)T, (uint64_t)ld16, (uint64_t)ld16, TC_BM);
  if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
  rc = make_tmap_f16(&tmB, loglam16, (uint64_t)EM_PB * Kpad, (uint64_t)ld16, (uint64_t)ld16, (uint32_t)BN);
  if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;

  EmissionTcParams p;
  p.T = T; p.K = K; p.Kpad = Kpad; p.BN = BN;
  p.n_kblocks = (int)((ld16 + TC_BK - 1) / TC_BK);
  p.n_mtiles = (int)((T + TC_BM - 1) / TC_BM);
  p.n_ntiles = n_ntiles;
  // no per-CTA rotation of the K-block order: every tile accumulates the neuron blocks in the same order, so
  // ll[t,:] is bit-identical wherever bin t sits in the launch -- time-sharded ranks recompute their neighbours'
  // halo bins and their seam checks compare messages at 1e-5 (a rotated order changes ll by ~3e-5 absolute)
  p.stagger = 0;
  p.idesc = make_idesc_f16(TC_BM, BN, 0, 0, 0);
  p.tmem_cols = pow2_cols(2 * BN);
  p.lam_sum = lam_sum; p.lgam = lgam; p.ma_latent = ma_latent; p.ll = ll; p.ldll = ldll;
  p.ep_nbuf = 0;
  cudaStream_t st = (cudaStream_t)stream;
  int dev = 0, sms = 0;
  PMG_CUDA_CHECK(cudaGetDevice(&dev));
  PMG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const size_t smem_max = 227 * 1024;

  // 256-row work units + TMA-store epilogue: needs 16-byte aligned rows of ll
  bool paired = (ldll & 3) == 0 && ((uintptr_t)ll & 15) == 0;
  // CTA pairs (cta_group::2): 512-row units, every log-rate tile shared by the two SMs of a TPC
  if (paired && (BN % 16) == 0 && T >= 4 * TC_BM) {
    const uint32_t stage_bytes = EM_MI * TC_A_BYTES + EM_PB * (BN / 2) * TC_BK * 2;
    const size_t fixed = 1024 /*align*/ + 256 /*barriers*/ + (size_t)((Kpad + 3) & ~3) * sizeof(float);
    // staging tiles per epilogue warp vs pipeline stages: two tiles unless that leaves fewer than three stages
    // (measured at the headline shape: 2 tiles / 3 stages 0.75 ms; forcing 2 or 3 tiles with 2 stages 0.83 ms)
    int nbuf = 2, stages = 0;
    for (; nbuf >= 1; --nbuf) {
      const size_t stg_bytes = (size_t)8 * nbuf * EP_BUF_BYTES;
      stages = fixed + stg_bytes < smem_max ? (int)((smem_max - fixed - stg_bytes) / stage_bytes) : 0;
      if (stages >= 3) break;
    }
    if (nbuf < 1) { nbuf = 1; }
    if (stages >= 2) {
      if (stages > 6) stages = 6;
      EmissionTcParams p2 = p;
      p2.stages = stages;
      p2.ep_nbuf = nbuf;
      p2.idesc = make_idesc_f16(2 * TC_BM, BN, 0, 0, 0);
      CUtensorMap tmBh, tmC32, tmC16;
      rc = make_tmap_f16(&tmBh, loglam16, (uint64_t)EM_PB * Kpad, (uint64_t)ld16, (uint64_t)ld16, (uint32_t)(BN / 2));
      if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
      rc = make_tmap_f32(&tmC32, ll, (uint64_t)T, (uint64_t)K, (uint64_t)ldll, 32, 32);
      if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
      rc = make_tmap_f32(&tmC16, ll, (uint64_t)T, (uint64_t)K, (uint64_t)ldll, 32, 16);
      if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
      const size_t smem = (size_t)stages * stage_bytes + (size_t)8 * nbuf * EP_BUF_BYTES + fixed;
      PMG_CUDA_CHECK(cudaFuncSetAttribute(emission_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      PMG_CUDA_CHECK(cudaFuncSetAttribute(emission_tc2_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 0));
      cudaLaunchConfig_t cfg = {};
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.blockDim = dim3(EM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st;
      cfg.attrs = attr; cfg.numAttrs = 1;
      cfg.gridDim = dim3((unsigned)(sms & ~1));
      // (the occupancy query costs tens of microseconds of host time: once per shared-memory size)
      static size_t occ_smem = 0;
      static int occ_clusters = 0, occ_dev = -1;
      static cudaError_t occ_err = cudaSuccess;
      if (occ_smem != smem || occ_dev != dev) {
        occ_dev = dev;
        occ_err = cudaOccupancyMaxActiveClusters(&occ_clusters, emission_tc2_kernel, &cfg);
        occ_smem = smem;
      }
      const int max_clusters = occ_clusters;
      const cudaError_t oe = occ_err;
      const int n_units2 = ((p.n_mtiles + 2 * EM_MI - 1) / (2 * EM_MI)) * p.n_ntiles;
      if (oe == cudaSuccess && max_clusters >= 1) {
        int n_cl = max_clusters < n_units2 ? max_clusters : n_units2;
        if (n_cl > sms / 2) n_cl = sms / 2;
        cfg.gridDim = dim3((unsigned)(2 * n_cl));
        PMG_CUDA_CHECK(cudaLaunchKernelEx(&cfg, emission_tc2_kernel, tmA, tmBh, tmC32, tmC16, p2));
        return PMG_OK;
      }
      (void)cudaGetLastError();          // no co-resident pair on this device/configuration: single-CTA kernel below
    }
  }
  if (paired) {
    const uint32_t stage_bytes = EM_MI * TC_A_BYTES + EM_PB * BN * TC_BK * 2;
    const size_t fixed = 1024 /*align*/ + 256 /*barriers*/ + (size_t)((Kpad + 3) & ~3) * sizeof(float);
    int nbuf = 2;
    int stages = 0;
    for (; nbuf >= 1; --nbuf) {
      const size_t stg_bytes = (size_t)8 * nbuf * EP_BUF_BYTES;
      stages = fixed + stg_bytes < smem_max ? (int)((smem_max - fixed - stg_bytes) / stage_bytes) : 0;
      if (stages >= 2) break;
    }
    if (stages < 2) {
      paired = false;
    } else {
      if (stages > 6) stages = 6;
      p.stages = stages;
      p.ep_nbuf = nbuf;
      CUtensorMap tmC32, tmC16;
      rc = make_tmap_f32(&tmC32, ll, (uint64_t)T, (uint64_t)K, (uint64_t)ldll, 32, 32);
      if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
      rc = make_tmap_f32(&tmC16, ll, (uint64_t)T, (uint64_t)K, (uint64_t)ldll, 32, 16);
      if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
      const size_t smem = (size_t)stages * stage_bytes + (size_t)8 * nbuf * EP_BUF_BYTES + fixed;
      PMG_CUDA_CHECK(cudaFuncSetAttribute(emission_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      const int n_units = ((p.n_mtiles + EM_MI - 1) / EM_MI) * p.n_ntiles;
      emission_tc_kernel<<<n_units < sms ? n_units : sms, EM_THREADS, smem, st>>>(tmA, tmB, tmC32, tmC16, p);
      PMG_LAUNCH_CHECK();
      return PMG_OK;
    }
  }
  // single-tile kernel with direct stores (any row pitch)
  {
    const uint32_t stage_bytes = TC_A_BYTES + EM_PB * BN * TC_BK * 2;
    int stages = (int)((225 * 1024) / stage_bytes);
    // measured on B200 at the headline shape: 2 stages 1.95 ms, 3 stages 2.08 ms
    if (stages > 2) stages = 2;
    if (stages < 2) return PMG_ERR_UNSUPPORTED_SHAPE;
    p.stages = stages;
    const size_t smem = (size_t)stages * stage_bytes + 1024 /*align*/ + 256 /*barriers*/;
    PMG_CUDA_CHECK(cudaFuncSetAttribute(emission_tc_kernel_v1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int n_tiles = p.n_mtiles * p.n_ntiles;
    emission_tc_kernel_v1<<<n_tiles < sms ? n_tiles : sms, TC_THREADS, smem, st>>>(tmA, tmB, p);
    PMG_LAUNCH_CHECK();
  }
  return PMG_OK;
}

// ---------------------------------------------------------------------------------------------
// time reduction: yw[k,n] = sum_t gamma[t,k] * y[t,n]   (both operands MN-major, time = UMMA K)
// accumulator tile: lanes = neurons (M = 128), columns = latent bins (N = BN, multiple of 64)
// ---------------------------------------------------------------------------------------------
namespace pmg {

constexpr int AT_BKT = 32;                       // time bins per pipeline stage
constexpr int AT_BOX_BYTES = AT_BKT * 128;       // one TMA box: 32 rows x 64 halves
constexpr int AT_PG = 2;                         // fp16 pieces of gamma

struct AtbTcParams {
  int64_t T, t_per_split;
  int64_t g_lo_row;  // row of the lo piece's first time bin in its tensor map (T: pieces stacked in one matrix; 0: own map)
  int K, N, BN, n_mtiles, n_ntiles, splits, stages;
  uint32_t tmem_cols;
  float* partial;    // [splits][K][N]
};

// One CTA owns TWO 128-neuron row tiles (two TMEM accumulators side by side) for one tile of latent bins and
// one time split, so that every posterior tile fetched from L2 feeds 256 output rows: the kernel is bound by
// the L2 -> shared-memory feed, not by the tensor pipe.
// PA = pieces of the row-side operand (1: exact fp16 counts; 2: hi/lo pieces, products hi*hi + hi*lo + lo*hi),
// FMT = 0 fp16, 1 bf16.
template <int PA, int FMT>
__global__ void __launch_bounds__(TC_THREADS, 1)
atb_tc_kernel(const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmY1,
              const __grid_constant__ CUtensorMap tmG, const __grid_constant__ CUtensorMap tmG1,
              const AtbTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int mp = blockIdx.x, nt = blockIdx.y, sp = blockIdx.z;
  const int n_mi = (2 * mp + 1 < p.n_mtiles) ? 2 : 1;          // row tiles of this CTA
  const int k_base = nt * p.BN;
  int bn = p.K - k_base;                         // columns of this tile, rounded up to the 64-wide atoms
  bn = (bn + 63) / 64 * 64;
  if (bn > p.BN) bn = p.BN;
  const int n_boxes_b = bn / 64;
  const uint32_t a_tile_bytes = 2 * AT_BOX_BYTES;              // 128 neurons x 32 time bins (one piece)
  const uint32_t a_bytes = 2 * PA * a_tile_bytes;
  const uint32_t b_piece_bytes = (uint32_t)(p.BN / 64) * AT_BOX_BYTES;
  const uint32_t stage_bytes = a_bytes + AT_PG * b_piece_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
  uint64_t* empty = full + p.stages;
  uint64_t* tfull = empty + p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmY); tma_prefetch_desc(&tmG); tma_prefetch_desc(&tmG1); }
  if (warp == 2) { tmem_alloc(tmem_slot, p.tmem_cols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t t_begin = (int64_t)sp * p.t_per_split;
  int64_t t_end = t_begin + p.t_per_split;
  if (t_end > p.T) t_end = p.T;
  const int n_tb = t_end > t_begin ? (int)((t_end - t_begin + AT_BKT - 1) / AT_BKT) : 0;
  const uint32_t tx_bytes = (uint32_t)(n_mi * PA) * a_tile_bytes + AT_PG * (uint32_t)n_boxes_b * AT_BOX_BYTES;

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tb = 0; tb < n_tb; ++tb) {
        mbar_wait(&empty[stage], phase ^ 1);
        uint8_t* sA = smem + (size_t)stage * stage_bytes;
        const int t0 = (int)(t_begin + (int64_t)tb * AT_BKT);
        mbar_arrive_expect_tx(&full[stage], tx_bytes);
        for (int mi = 0; mi < n_mi; ++mi) {
          const int m0 = (2 * mp + mi) * TC_BM;
#pragma unroll
          for (int pa = 0; pa < PA; ++pa) {       // one tensor map per piece: rows past T are zero-filled
            const CUtensorMap* tm = pa == 0 ? &tmY : &tmY1;
            uint8_t* dst = sA + (mi * PA + pa) * a_tile_bytes;
            tma_load_2d(dst, tm, &full[stage], m0, t0);
            tma_load_2d(dst + AT_BOX_BYTES, tm, &full[stage], m0 + 64, t0);
          }
        }
        for (int pc = 0; pc < AT_PG; ++pc)
          for (int b = 0; b < n_boxes_b; ++b)
            tma_load_2d(sA + a_bytes + pc * b_piece_bytes + b * AT_BOX_BYTES, pc == 0 ? &tmG : &tmG1, &full[stage],
                        k_base + b * 64, (int)(pc * p.g_lo_row) + t0);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_f16(TC_BM, bn, 1, 1, FMT);
      int stage = 0; uint32_t phase = 0;
      for (int tb = 0; tb < n_tb; ++tb) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        const uint32_t sA = smem_u32(smem + (size_t)stage * stage_bytes);
        for (int mi = 0; mi < n_mi; ++mi) {
#pragma unroll
          for (int pa = 0; pa < PA; ++pa) {
#pragma unroll
            for (int pc = 0; pc < AT_PG; ++pc) {
              if (pa + pc > 1) continue;          // lo*lo is below the kept precision
              const uint32_t sB = sA + a_bytes + pc * b_piece_bytes;
#pragma unroll
              for (int k = 0; k < AT_BKT / 16; ++k) {
                // MN-major: atoms along M/N are one TMA box apart (LBO), 8-row atoms along time 1024 B apart (SBO)
                const uint64_t ad = make_smem_desc(sA + (mi * PA + pa) * a_tile_bytes + k * 2048, AT_BOX_BYTES, 1024);
                const uint64_t bd = make_smem_desc(sB + k * 2048, AT_BOX_BYTES, 1024);
                mma_f16_ss(tmem_base + (uint32_t)(mi * p.BN), ad, bd, idesc, (tb | pa | pc | k) != 0);
              }
            }
          }
        }
        mma_commit(&empty[stage]);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      mma_commit(tfull);
    }
  } else if (warp >= 4) {
    const int q = warp & 3;
    float* out = p.partial + (size_t)sp * p.K * p.N;
    if (n_tb > 0) {
      mbar_wait(tfull, 0);
      tc_fence_after();
    }
    for (int mi = 0; mi < n_mi; ++mi) {
      const int n = (2 * mp + mi) * TC_BM + q * 32 + lane;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(mi * p.BN);
      for (int c0 = 0; c0 < bn; c0 += 16) {
        uint32_t r[16];
        if (n_tb > 0) {
          tmem_ld_x16(taddr + c0, r);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) r[j] = 0u;
        }
        if (n < p.N) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const int k = k_base + c0 + j;
            if (k < p.K) out[(size_t)k * p.N + n] = __uint_as_float(r[j]);   // lanes = consecutive neurons: coalesced
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, p.tmem_cols); }
}

// [T,K] fp32 -> two bf16 pieces [2][T][ld16] (hi + lo = 16 significant bits, fp32 exponent range), zero padded
__global__ void split_bf16_kernel(int64_t T, int K, const float* __restrict__ src, int64_t lds,
                                  __nv_bfloat16* __restrict__ dst, int64_t ld16) {
  const int64_t total = T * ld16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / ld16;
    const int k = (int)(i - t * ld16);
    const float v = k < K ? src[(size_t)t * lds + k] : 0.f;
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    dst[i] = h;
    dst[total + i] = __float2bfloat16_rn(v - __bfloat162float(h));
  }
}

// vectorised variant (K % 8 == 0, 16-byte aligned rows): 8 elements per thread, two 16-byte loads, two 16-byte stores
// per piece; one warp-sized stripe of a row at a time.  HALF = 1: fp16 pieces, else bf16.
template <int HALF>
__global__ void __launch_bounds__(256) split_pieces_vec_kernel(int64_t T, int K8, const float* __restrict__ src,
                                                               int64_t lds, uint16_t* __restrict__ dst, int64_t ld16) {
  const int64_t total = T * (int64_t)K8;          // groups of 8 elements
  const size_t piece = (size_t)T * ld16;
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < total; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = g / K8;
    const int k = (int)(g - t * K8) * 8;
    const float4* sp = reinterpret_cast<const float4*>(src + (size_t)t * lds + k);
    const float4 a = __ldcs(sp), b = __ldcs(sp + 1);
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint16_t hi[8], lo[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      if (HALF) {
        const __half h = __float2half_rn(v[e]);
        hi[e] = __half_as_ushort(h);
        lo[e] = __half_as_ushort(__float2half_rn(v[e] - __half2float(h)));
      } else {
        const __nv_bfloat16 h = __float2bfloat16_rn(v[e]);
        hi[e] = __bfloat16_as_ushort(h);
        lo[e] = __bfloat16_as_ushort(__float2bfloat16_rn(v[e] - __bfloat162float(h)));
      }
    }
    uint4 H, L;
    H.x = hi[0] | ((uint32_t)hi[1] << 16); H.y = hi[2] | ((uint32_t)hi[3] << 16);
    H.z = hi[4] | ((uint32_t)hi[5] << 16); H.w = hi[6] | ((uint32_t)hi[7] << 16);
    L.x = lo[0] | ((uint32_t)lo[1] << 16); L.y = lo[2] | ((uint32_t)lo[3] << 16);
    L.z = lo[4] | ((uint32_t)lo[5] << 16); L.w = lo[6] | ((uint32_t)lo[7] << 16);
    uint16_t* o = dst + (size_t)t * ld16 + k;
    *reinterpret_cast<uint4*>(o) = H;
    *reinterpret_cast<uint4*>(o + piece) = L;
  }
}

static bool split_vec_ok(int K, const void* src, int64_t lds, const void* dst, int64_t ld16) {
  return (K % 8) == 0 && K == ld16 && (lds % 4) == 0 && (((uintptr_t)src | (uintptr_t)dst) & 15) == 0;
}

// posterior [T,K] fp32 -> two fp16 pieces [2][T][ld16] (hi + lo), zero padded
__global__ void split_f16_kernel(int64_t T, int K, const float* __restrict__ src, int64_t lds,
                                 __half* __restrict__ dst, int64_t ld16) {
  const int64_t total = T * ld16;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t t = i / ld16;
    const int k = (int)(i - t * ld16);
    const float v = k < K ? src[(size_t)t * lds + k] : 0.f;
    const __half h = __float2half_rn(v);
    dst[i] = h;
    dst[total + i] = __float2half_rn(v - __half2float(h));
  }
}

__global__ void split_reduce_kernel_tc(int splits, int64_t MN, const float* __restrict__ partial,
                                       float* __restrict__ C) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= MN) return;
  double s = 0.0;
  for (int z = 0; z < splits; ++z) s += (double)partial[(size_t)z * MN + i];
  C[i] = (float)s;
}

static void atb_tc_plan(int64_t T, int K, int N, int& BN, int& n_mtiles, int& n_ntiles, int& splits,
                        int64_t& t_per_split) {
  BN = K >= 256 ? 256 : (K + 63) / 64 * 64;
  n_ntiles = (K + BN - 1) / BN;
  n_mtiles = (N + TC_BM - 1) / TC_BM;
  const int tiles = ((n_mtiles + 1) / 2) * n_ntiles;   // a CTA owns a pair of row tiles
  splits = 148 / tiles;
  if (splits < 1) splits = 1;
  const int64_t max_splits = (T + 4 * AT_BKT - 1) / (4 * AT_BKT);
  if (splits > max_splits) splits = (int)max_splits;
  if (splits < 1) splits = 1;
  t_per_split = ((T + splits - 1) / splits + AT_BKT - 1) / AT_BKT * AT_BKT;
  splits = (int)((T + t_per_split - 1) / t_per_split);
}

}  // namespace pmg

extern "C" int pmg_split_f16(int64_t T, int K, const float* src, int64_t lds, void* dst16, int64_t ld16,
                             pmg_stream_t stream) {
  if (T <= 0 || K <= 0 || !src || !dst16 || lds < K || ld16 < K || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  if (pmg::split_vec_ok(K, src, lds, dst16, ld16))
    pmg::split_pieces_vec_kernel<1><<<148 * 16, 256, 0, (cudaStream_t)stream>>>(T, K / 8, src, lds, (uint16_t*)dst16, ld16);
  else
    pmg::split_f16_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(T, K, src, lds, (__half*)dst16, ld16);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int64_t pmg_atb_f16_workspace_bytes(int64_t T, int K, int N) {
  if (T <= 0 || K <= 0 || N <= 0) return 0;
  int BN, nm, nn, splits; int64_t tps;
  pmg::atb_tc_plan(T, K, N, BN, nm, nn, splits, tps);
  return (int64_t)splits * K * N * (int64_t)sizeof(float);
}

extern "C" int pmg_split_bf16(int64_t T, int K, const float* src, int64_t lds, void* dst16, int64_t ld16,
                              pmg_stream_t stream) {
  if (T <= 0 || K <= 0 || !src || !dst16 || lds < K || ld16 < K || (ld16 & 7)) return PMG_ERR_BAD_ARG;
  if (pmg::split_vec_ok(K, src, lds, dst16, ld16))
    pmg::split_pieces_vec_kernel<0><<<148 * 16, 256, 0, (cudaStream_t)stream>>>(T, K / 8, src, lds, (uint16_t*)dst16, ld16);
  else
    pmg::split_bf16_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(T, K, src, lds, (__nv_bfloat16*)dst16, ld16);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

static int atb_pieces_launch(int64_t T, int K, int N, const void* g16, const void* g16_lo, int64_t ldg,
                             const void* y16, const void* y16_lo, int64_t ldy16, int fmt, float* yw, void* workspace,
                             int64_t workspace_bytes, pmg_stream_t stream);

extern "C" int pmg_atb_f16(int64_t T, int K, int N, const void* g16, int64_t ldg, const void* y16, int64_t ldy16,
                           float* yw, void* workspace, int64_t workspace_bytes, pmg_stream_t stream) {
  return atb_pieces_launch(T, K, N, g16, nullptr, ldg, y16, nullptr, ldy16, 0, yw, workspace, workspace_bytes, stream);
}

// out[k,n] = sum_t G[t,k] * Y[t,n] with BOTH operands given as two bf16 pieces ([2][T][ld], hi then lo):
// three tensor-core products (hi*hi + hi*lo + lo*hi), fp32 accumulation, relative error ~2^-16.
// Same workspace as pmg_atb_f16 (pmg_atb_f16_workspace_bytes).
extern "C" int pmg_atb_bf16x2(int64_t T, int K, int N, const void* g16, int64_t ldg, const void* y16, int64_t ldy16,
                              float* out, void* workspace, int64_t workspace_bytes, pmg_stream_t stream) {
  if (!y16 || T <= 0) return PMG_ERR_BAD_ARG;
  const char* lo = (const char*)y16 + (size_t)T * (size_t)ldy16 * 2;
  return atb_pieces_launch(T, K, N, g16, nullptr, ldg, y16, lo, ldy16, 1, out, workspace, workspace_bytes, stream);
}

// Same product with every piece behind its own pointer (rows of T bins, common leading dimension per operand): the
// pieces the backward scan writes for the transition counts (pmg_backward_xi16) are used in place, at a row offset.
extern "C" int pmg_atb_bf16x2_pieces(int64_t T, int K, int N, const void* g_hi, const void* g_lo, int64_t ldg,
                                     const void* y_hi, const void* y_lo, int64_t ldy16, float* out, void* workspace,
                                     int64_t workspace_bytes, pmg_stream_t stream) {
  if (!g_hi || !g_lo || !y_hi || !y_lo || T <= 0) return PMG_ERR_BAD_ARG;
  return atb_pieces_launch(T, K, N, g_hi, g_lo, ldg, y_hi, y_lo, ldy16, 1, out, workspace, workspace_bytes, stream);
}

static int atb_pieces_launch(int64_t T, int K, int N, const void* g16, const void* g16_lo, int64_t ldg,
                             const void* y16, const void* y16_lo, int64_t ldy16, int fmt, float* yw, void* workspace,
                             int64_t workspace_bytes, pmg_stream_t stream) {
  using namespace pmg;
  if (T <= 0 || K <= 0 || N <= 0 || !g16 || !y16 || !yw) return PMG_ERR_BAD_ARG;
  if (ldg < K || (ldg & 7) || ldy16 < N || (ldy16 & 7)) return PMG_ERR_BAD_ARG;
  if (((uintptr_t)g16 & 15) || ((uintptr_t)y16 & 15) || ((uintptr_t)g16_lo & 15)) return PMG_ERR_ALIGNMENT;
  if ((int64_t)AT_PG * T > ((int64_t)1 << 31) - 256) return PMG_ERR_UNSUPPORTED_SHAPE;
  AtbTcParams p;
  atb_tc_plan(T, K, N, p.BN, p.n_mtiles, p.n_ntiles, p.splits, p.t_per_split);
  if (!workspace || workspace_bytes < (int64_t)p.splits * K * N * (int64_t)sizeof(float)) return PMG_ERR_WORKSPACE;
  p.T = T; p.K = K; p.N = N; p.partial = (float*)workspace;
  const int PA = y16_lo ? 2 : 1;
  if (y16_lo && ((uintptr_t)y16_lo & 15)) return PMG_ERR_ALIGNMENT;
  const uint32_t stage_bytes = 4 * PA * AT_BOX_BYTES + AT_PG * (p.BN / 64) * AT_BOX_BYTES;
  int stages = (int)((200 * 1024) / stage_bytes);
  if (stages > 8) stages = 8;
  if (stages < 2) return PMG_ERR_UNSUPPORTED_SHAPE;
  p.stages = stages;
  p.tmem_cols = pow2_cols(2 * p.BN);

  CUtensorMap tmY, tmY1, tmG, tmG1;
  // inner (contiguous) dimension = neurons / latent bins, outer = time; box = 32 time rows x 64 columns
  // (fp16 and bf16 share the 2-byte tensor-map geometry; the data type only matters to the MMA descriptor)
  int rc = make_tmap_f16(&tmY, y16, (uint64_t)T, (uint64_t)ldy16, (uint64_t)ldy16, AT_BKT);
  if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
  rc = make_tmap_f16(&tmY1, y16_lo ? y16_lo : y16, (uint64_t)T, (uint64_t)ldy16, (uint64_t)ldy16, AT_BKT);
  if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
  // posterior-side pieces: stacked [2][T][ldg] in one matrix (lo piece T rows further down), or one matrix each
  rc = make_tmap_f16(&tmG, g16, (uint64_t)(g16_lo ? 1 : AT_PG) * T, (uint64_t)ldg, (uint64_t)ldg, AT_BKT);
  if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
  tmG1 = tmG;
  p.g_lo_row = T;
  if (g16_lo) {
    rc = make_tmap_f16(&tmG1, g16_lo, (uint64_t)T, (uint64_t)ldg, (uint64_t)ldg, AT_BKT);
    if (rc) return PMG_ERR_UNSUPPORTED_SHAPE;
    p.g_lo_row = 0;
  }
  const size_t smem = (size_t)stages * stage_bytes + 1024 + 256;
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid((p.n_mtiles + 1) / 2, p.n_ntiles, p.splits);
  if (PA == 1 && fmt == 0) {
    PMG_CUDA_CHECK(cudaFuncSetAttribute(atb_tc_kernel<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    atb_tc_kernel<1, 0><<<grid, TC_THREADS, smem, st>>>(tmY, tmY1, tmG, tmG1, p);
  } else if (PA == 2 && fmt == 1) {
    PMG_CUDA_CHECK(cudaFuncSetAttribute(atb_tc_kernel<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    atb_tc_kernel<2, 1><<<grid, TC_THREADS, smem, st>>>(tmY, tmY1, tmG, tmG1, p);
  } else {
    return PMG_ERR_BAD_ARG;
  }
  PMG_LAUNCH_CHECK();
  const int64_t MN = (int64_t)K * N;
  split_reduce_kernel_tc<<<cdiv(MN, 256), 256, 0, st>>>(p.splits, MN, p.partial, yw);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

// legacy hooks of pmg_atb (fp32 operands): the tensor-core path needs fp16 pieces, see pmg_atb_f16
int64_t pmg_atb_tc_workspace_bytes(int64_t, int, int) { return 0; }
int pmg_atb_tc_launch(int64_t, int, int, const float*, int64_t, const float*, int64_t, float*, int64_t, void*,
                      int64_t, cudaStream_t) {
  return PMG_ERR_UNSUPPORTED_SHAPE;
}
