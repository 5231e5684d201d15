// Bulk-copy (TMA 1-D, cp.async.bulk + mbarrier) variants of the forward / backward chain kernels.
//
// Same recursion as fwd_kernel / bwd_kernel (pmg_scan.cu) for the headline case — one warp per
// chain, Toeplitz "move" kernel with band half width <= WT, K % 8 == 0 — restructured for
// throughput:
//   * every T-sized array is streamed through shared memory with whole-row asynchronous bulk
//     copies: inputs (ll rows, alpha rows) arrive in an R-deep ring with one mbarrier per slot,
//     issued R steps ahead by lane 0; outputs (alpha rows, fp16 posterior pieces) are staged in
//     shared memory and leave as bulk stores (double buffered, cp.async.bulk.wait_group.read);
//   * shared-memory rows are padded to 32*Q floats, so the time loop has no bounds predicates;
//   * the per-step normaliser is applied one step late (folded into the likelihood factor), which
//     takes the warp reduction and the reciprocal off the loop-carried dependency chain.
// Included by pmg_scan.cu (needs Geo, band_apply, chain_range, FwdParams, BwdParams).
#pragma once
#include <cuda_bf16.h>

#include "pmg_tc.cuh"

namespace pmg {

__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(tc::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(tc::smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_store(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
               ::"l"(gdst), "r"(tc::smem_u32(smem_src)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__host__ __device__ inline int round4(int v) { return (v + 3) & ~3; }

template <int Q, int WT>
struct BulkGeo {
  using Ge = Geo<Q, 1, WT>;
  static constexpr int KP = 32 * Q;                       // padded row length in shared memory
  __host__ __device__ static int exf() { return round4(Ge::buf_floats(0)); }
  // floats per chain: mbarriers | exchange x2 | input ring | output staging x2
  // OB = number of output staging buffers (2: store of step t overlaps step t+1; 1: smaller footprint)
  __host__ __device__ static int fwd_chain_floats(int R, int OB) {
    return round4(2 * R) + 2 * exf() + R * KP + OB * 2 * KP;
  }
  __host__ __device__ static int bwd_chain_floats(int R, int OB) {
    return round4(2 * R) + 2 * exf() + R * 3 * KP + OB * KP + KP;   // + one fp32 row: transpose staging
  }
};

constexpr float kLog2e = 1.4426950408889634f;

// ============================================================================
// forward, bulk I/O
// ============================================================================
template <int Q, int WT, int NW, int OB>
__global__ void __launch_bounds__(32 * NW, 1) fwd_bulk_kernel(const FwdParams p, const int R) {
  using Ge = Geo<Q, 1, WT>;
  using BG = BulkGeo<Q, WT>;
  constexpr int KP = BG::KP;
  extern __shared__ __align__(16) float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, NW)) return;
  const int K = c.tr.K, W = c.tr.W;
  const int grp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int bar_id = 1 + grp;
  const int x0 = lane * Q;

  const int exf = BG::exf();
  float* base = smem + (size_t)grp * BG::fwd_chain_floats(R, OB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base);
  float* exch = base + round4(2 * R);
  float* ring = exch + 2 * exf;                 // R rows of KP floats; columns >= K stay -inf
  float* outb = ring + (size_t)R * KP;          // 2 buffers x (move row KP | jump row KP)
  for (int i = lane; i < 2 * exf; i += 32) exch[i] = 0.f;
  for (int i = lane; i < R * KP; i += 32) ring[i] = -INFINITY;
  if (lane == 0) {
    for (int s = 0; s < R; ++s) tc::mbar_init(&bars[s], 1);
    tc::fence_barrier_init();
  }
  fence_proxy_async();
  __syncthreads();

  ChainRange cr;
  if (!chain_range<NW>(c, grp, cr)) return;

  float tp[2 * WT + 1];
#pragma unroll
  for (int j = 0; j <= 2 * WT; ++j) {
    const int d = j >= WT ? j - WT : WT - j;
    tp[j] = d <= W ? __ldg(c.tr.taps + d) : 0.f;
  }
  // a0 = (M00*v0 + M10*v1)/z folded into two per-bin constants
  float m0z[Q], m1z[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const float iz = (x0 + q < K) ? __ldg(c.tr.inv_z + x0 + q) : 0.f;
    m0z[q] = c.tr.M00 * iz;
    m1z[q] = c.tr.M10 * iz;
  }
  const float M01 = c.tr.M01, M11 = c.tr.M11;
  const float invK = 1.f / (float)K;
  const float sc2 = c.scale * kLog2e;            // exp(s*(ll-m)) = exp2(sc2*ll - sc2*m)

  // ---- initial carry (same rules as fwd_kernel): v = alpha_{t0-1} (normalised), inv_prev = 1
  int64_t t0;
  float v0[Q], v1[Q];
  const float* src = fwd_start<true>(c, cr, p, t0, K);
  float S0 = 0.f, S1 = 0.f;
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const bool ok = x0 + q < K;
    v0[q] = ok ? (src ? src[x0 + q] : 0.5f * invK) : 0.f;
    v1[q] = ok ? (src ? src[K + x0 + q] : 0.5f * invK) : 0.f;
    S0 += v0[q];
    S1 += v1[q];
  }
  S0 = warp_sum(S0); S1 = warp_sum(S1);
  if (!(S0 + S1 > 0.f) || !(S0 + S1 < 3.0e38f)) {
    // unusable initial message (all zero / non-finite): fall back to the uniform one
#pragma unroll
    for (int q = 0; q < Q; ++q) { v0[q] = (x0 + q < K) ? 0.5f * invK : 0.f; v1[q] = v0[q]; }
    S0 = 0.5f; S1 = 0.5f;
  }
  float inv_prev = 1.f / (S0 + S1);

  // ---- fill the input ring
  const uint32_t row_bytes = (uint32_t)K * 4;
  const int64_t n_steps = cr.t_end - t0;
  if (lane == 0) {
    for (int j = 0; j < R && j < n_steps; ++j) {
      tc::mbar_arrive_expect_tx(&bars[j], row_bytes);
      bulk_load(ring + (size_t)j * KP, c.ll + (size_t)(t0 + j) * c.ldll, row_bytes, &bars[j]);
    }
  }

  int par = 0, slot = 0, out_par = 0;
  uint32_t ring_phase = 0;
  for (int64_t i = 0; i < n_steps; ++i) {
    const int64_t t = t0 + i;
    if (lane == 0) bulk_wait_read<OB - 1>();     // staging buffer `out_par` is free again
    tc::mbar_wait(&bars[slot], ring_phase);
    float Lc[Q];
    float m = -INFINITY;
    {
      const float* row = ring + (size_t)slot * KP + x0;
#pragma unroll
      for (int q = 0; q < Q; ++q) { Lc[q] = row[q]; m = fmaxf(m, Lc[q]); }
    }
    // carried message -> exchange buffer (the loop-carried chain starts here)
    float a0[Q], pr0[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) a0[q] = fmaf(m0z[q], v0[q], m1z[q] * v1[q]);
    band_apply<Q, 1, WT>(a0, pr0, exch + par * exf, lane, tp, nullptr, nullptr, 0, W, K, bar_id);
    par ^= 1;
    // every lane has consumed ring[slot] (warp sync inside band_apply): refill it R steps ahead
    if (lane == 0 && i + R < n_steps) {
      fence_proxy_async();
      tc::mbar_arrive_expect_tx(&bars[slot], row_bytes);
      bulk_load(ring + (size_t)slot * KP, c.ll + (size_t)(t + R) * c.ldll, row_bytes, &bars[slot]);
    }
    if (++slot == R) { slot = 0; ring_phase ^= 1; }

    // likelihood factor with the previous normaliser folded in (off the carried chain)
    m = warp_max(m);
    const float msc = m * sc2;
#pragma unroll
    for (int q = 0; q < Q; ++q) Lc[q] = exp2f(fmaf(Lc[q], sc2, -msc)) * inv_prev;   // pad columns: exp2(-inf) = 0
    const float p1 = (M01 * S0 + M11 * S1) * invK;
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      v0[q] = pr0[q] * Lc[q];
      v1[q] = p1 * Lc[q];
      s0 += v0[q];
      s1 += v1[q];
    }
    S0 = warp_sum(s0); S1 = warp_sum(s1);
    const float cn = S0 + S1;                   // c_t = sum of prior x likelihood
    inv_prev = 1.f / cn;

    if (t >= cr.t_begin) {
      float* ob = outb + (size_t)out_par * 2 * KP;
#pragma unroll
      for (int q = 0; q < Q; ++q) { ob[x0 + q] = v0[q] * inv_prev; ob[KP + x0 + q] = v1[q] * inv_prev; }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) {
        float* dst = p.alpha + (size_t)t * 2 * K;
        bulk_store(dst, ob, row_bytes);
        bulk_store(dst + K, ob + KP, row_bytes);
        bulk_commit();
        p.lmr[t] = logf(cn) + c.scale * m;
      }
      out_par = (out_par + 1) % OB;
    } else if (t == cr.t_begin - 1 && p.halo_state) {
      float* o = p.halo_state + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (x0 + q < K) { o[x0 + q] = v0[q] * inv_prev; o[K + x0 + q] = v1[q] * inv_prev; }
    }
    if (p.warm_out && t == cr.t_end - halo_next_of(c, cr.s + 1) - 1 && (cr.s + 1 < c.n_chain || !c.right_exact)) {
      float* o = p.warm_out + (size_t)(cr.s + 1) * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (x0 + q < K) { o[x0 + q] = v0[q] * inv_prev; o[K + x0 + q] = v1[q] * inv_prev; }
    }
  }
  if (lane == 0) bulk_wait_read<0>();
}

// ============================================================================
// backward, bulk I/O (ll and alpha rows in, fp16 posterior pieces out; the optional fp32
// outputs of the last EM iteration / decode are written directly)
// ============================================================================
template <int Q, int WT, int NW, int OB>
__global__ void __launch_bounds__(32 * NW, 1) bwd_bulk_kernel(const BwdParams p, const int R) {
  using Ge = Geo<Q, 1, WT>;
  using BG = BulkGeo<Q, WT>;
  constexpr int KP = BG::KP;
  extern __shared__ __align__(16) float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, NW)) return;
  const int K = c.tr.K, W = c.tr.W;
  const int grp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int bar_id = 1 + grp;
  const int x0 = lane * Q;

  const int exf = BG::exf();
  float* base = smem + (size_t)grp * BG::bwd_chain_floats(R, OB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base);
  float* exch = base + round4(2 * R);
  float* ring = exch + 2 * exf;                      // slot: [ll KP | alpha move KP | alpha jump KP]
  __half* outh = reinterpret_cast<__half*>(ring + (size_t)R * 3 * KP);   // 2 buffers x (hi KP | lo KP) halves
  float* trow = ring + (size_t)R * 3 * KP + (size_t)OB * KP;             // fp32 row: lane-blocked -> coalesced
  // fp32 output rows (gamma, gamma_lat, r: last EM iteration / decode): each lane owns Q consecutive latent
  // bins, so direct stores would scatter 4-byte pieces; the row goes through shared memory and leaves as
  // 16-byte stores of consecutive lanes (K % 4 == 0 and 16-byte aligned rows; otherwise scalar, still coalesced)
  const bool vec_rows = (K & 3) == 0;
  auto store_row = [&](float* dst, const float (&v)[Q], float scale) {
#pragma unroll
    for (int q = 0; q < Q; ++q) trow[x0 + q] = v[q] * scale;
    __syncwarp();
    if (vec_rows && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
      for (int j = lane * 4; j < K; j += 128)
        *reinterpret_cast<float4*>(dst + j) = *reinterpret_cast<const float4*>(trow + j);
    } else {
      for (int j = lane; j < K; j += 32) dst[j] = trow[j];
    }
    __syncwarp();
  };
  // bf16 hi/lo pieces of a [K] row (operands of the transition-count GEMM, rounding as pmg_split_bf16): staged in
  // the same shared row (KP bf16 hi | KP bf16 lo), written as 16-byte stores of consecutive lanes (K % 8 == 0)
  auto store_row_bf16 = [&](uint16_t* dst_hi, uint16_t* dst_lo, const float (&v)[Q], float scale) {
    __nv_bfloat16* th = reinterpret_cast<__nv_bfloat16*>(trow);
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const float f = v[q] * scale;
      const __nv_bfloat16 h = __float2bfloat16_rn(f);
      th[x0 + q] = h;
      th[KP + x0 + q] = __float2bfloat16_rn(f - __bfloat162float(h));
    }
    __syncwarp();
    for (int j = lane; j < K / 8; j += 32) {
      reinterpret_cast<uint4*>(dst_hi)[j] = reinterpret_cast<const uint4*>(th)[j];
      reinterpret_cast<uint4*>(dst_lo)[j] = reinterpret_cast<const uint4*>(th + KP)[j];
    }
    __syncwarp();
  };
  for (int i = lane; i < 2 * exf; i += 32) exch[i] = 0.f;
  for (int i = lane; i < R * 3 * KP; i += 32) ring[i] = ((i / KP) % 3 == 0) ? -INFINITY : 0.f;
  if (lane == 0) {
    for (int s = 0; s < R; ++s) tc::mbar_init(&bars[s], 1);
    tc::fence_barrier_init();
  }
  fence_proxy_async();
  __syncthreads();

  ChainRange cr;
  if (!chain_range<NW>(c, grp, cr)) return;

  float tp[2 * WT + 1];
#pragma unroll
  for (int j = 0; j <= 2 * WT; ++j) {
    const int d = j >= WT ? j - WT : WT - j;
    tp[j] = d <= W ? __ldg(c.tr.taps + d) : 0.f;
  }
  // beta_t[d,x] = M[d,0]*w0[x]/z[x] + M[d,1]*w1
  float m0z[Q], m1z[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const float iz = (x0 + q < K) ? __ldg(c.tr.inv_z + x0 + q) : 0.f;
    m0z[q] = c.tr.M00 * iz;
    m1z[q] = c.tr.M10 * iz;
  }
  const float M01 = c.tr.M01, M11 = c.tr.M11;
  const float invK = 1.f / (float)K;
  const float sc2 = c.scale * kLog2e;

  int64_t t_hi;
  const float* init = bwd_start<true>(c, cr, p, t_hi, K);

  // carried: unnormalised beta b (of the bin handled last), its normaliser inv_prev, its likelihood
  // factor Lb, and RLu = sum_x Lb*b1 (unnormalised jump-state sum)
  float b0[Q], b1[Q], Lb[Q], tw_acc[Q];
  float inv_prev = 1.f, RLu = 0.f;
#pragma unroll
  for (int q = 0; q < Q; ++q) { b0[q] = 0.f; b1[q] = 0.f; Lb[q] = 0.f; tw_acc[q] = 0.f; }

  // ---- input ring: step i handles bin t_hi - i; alpha is needed for bins <= t_end
  const uint32_t row_bytes = (uint32_t)K * 4;
  const int64_t n_steps = t_hi - cr.t_begin + 1;
  auto issue = [&](int s, int64_t t) {
    const bool need_a = t <= cr.t_end;
    tc::mbar_arrive_expect_tx(&bars[s], need_a ? 3 * row_bytes : row_bytes);
    float* dst = ring + (size_t)s * 3 * KP;
    bulk_load(dst, c.ll + (size_t)t * c.ldll, row_bytes, &bars[s]);
    if (need_a) {
      bulk_load(dst + KP, p.alpha + (size_t)t * 2 * K, row_bytes, &bars[s]);
      bulk_load(dst + 2 * KP, p.alpha + (size_t)t * 2 * K + K, row_bytes, &bars[s]);
    }
  };
  if (lane == 0) {
    for (int j = 0; j < R && j < n_steps; ++j) issue(j, t_hi - j);
  }

  int par = 0, slot = 0, out_par = 0;
  uint32_t ring_phase = 0;
  for (int64_t i = 0; i < n_steps; ++i) {
    const int64_t t = t_hi - i;
    const bool use_alpha = t <= cr.t_end;
    if (lane == 0) bulk_wait_read<OB - 1>();
    tc::mbar_wait(&bars[slot], ring_phase);
    const float* row = ring + (size_t)slot * 3 * KP + x0;

    // ---- unnormalised beta_t (carried chain: b -> exchange -> band -> b)
    float r0[Q], r1[Q];
    if (i == 0) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const bool ok = x0 + q < K;
        b0[q] = ok ? (init ? init[x0 + q] : 1.f) : 0.f;
        b1[q] = ok ? (init ? init[K + x0 + q] : 1.f) : 0.f;
        r0[q] = 0.f; r1[q] = 0.f;
      }
      {
        // unusable initial message (all zero / non-finite): fall back to the all-ones one
        float sb = 0.f;
#pragma unroll
        for (int q = 0; q < Q; ++q) sb += b0[q] + b1[q];
        sb = warp_sum(sb);
        if (!(sb > 0.f) || !(sb < 3.0e38f)) {
#pragma unroll
          for (int q = 0; q < Q; ++q) { b0[q] = (x0 + q < K) ? 1.f : 0.f; b1[q] = b0[q]; }
        }
      }
      __syncwarp();
    } else {
      float w0[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) { r0[q] = Lb[q] * b0[q]; r1[q] = Lb[q] * b1[q]; }   // Lb carries 1/normaliser
      band_apply<Q, 1, WT>(r0, w0, exch + par * exf, lane, tp, nullptr, nullptr, 0, W, K, bar_id);
      par ^= 1;
      const float w1 = RLu * inv_prev * invK;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const bool ok = x0 + q < K;
        b0[q] = fmaf(m0z[q], w0[q], ok ? M01 * w1 : 0.f);
        b1[q] = fmaf(m1z[q], w0[q], ok ? M11 * w1 : 0.f);
      }
    }

    // ---- likelihood factor of this bin, normaliser, posterior
    float Lc[Q];
    float m = -INFINITY;
#pragma unroll
    for (int q = 0; q < Q; ++q) { Lc[q] = row[q]; m = fmaxf(m, Lc[q]); }
    m = warp_max(m);
    const float msc = m * sc2;
#pragma unroll
    for (int q = 0; q < Q; ++q) Lc[q] = exp2f(fmaf(Lc[q], sc2, -msc));
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    float g0[Q], g1[Q];
    if (use_alpha) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        g0[q] = row[KP + q] * b0[q];
        g1[q] = row[2 * KP + q] * b1[q];
        s0 += g0[q];
        s1 += g1[q];
        s2 = fmaf(Lc[q], b1[q], s2);
      }
    } else {
#pragma unroll
      for (int q = 0; q < Q; ++q) { g0[q] = 0.f; g1[q] = 0.f; s0 += b0[q]; s1 += b1[q]; s2 = fmaf(Lc[q], b1[q], s2); }
    }
    if (p.xa_hi && t < cr.t_end) {              // alpha_t as bf16 pieces, while its row is still in the ring
      float av[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) av[q] = row[KP + q];
      store_row_bf16(p.xa_hi + (size_t)t * p.ld_x, p.xa_lo + (size_t)t * p.ld_x, av, 1.f);
#pragma unroll
      for (int q = 0; q < Q; ++q) av[q] = row[2 * KP + q];
      store_row_bf16(p.xa_hi + (size_t)t * p.ld_x + K, p.xa_lo + (size_t)t * p.ld_x + K, av, 1.f);
    }
    // all lanes are done with ring[slot]: refill it R steps ahead
    __syncwarp();
    if (lane == 0 && i + R < n_steps) {
      fence_proxy_async();
      issue(slot, t - R);
    }
    if (++slot == R) { slot = 0; ring_phase ^= 1; }

    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2);
    const float inv = 1.f / (s0 + s1);
    const float r_scale = inv;                       // r_{t+1} = Lb*b_{t+1}*inv_prev (in Lb) * inv
    inv_prev = inv;
    RLu = s2;
#pragma unroll
    for (int q = 0; q < Q; ++q) Lb[q] = Lc[q] * inv;

    if (t < cr.t_end) {
      float* g = p.gamma ? p.gamma + (size_t)t * 2 * K : nullptr;
      float* gl_ = p.gamma_lat ? p.gamma_lat + (size_t)t * K : nullptr;
      __half* oh = outh + (size_t)out_par * 2 * KP;
      float gsum[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const float ga = g0[q] * inv, gb = g1[q] * inv;
        const float gs = ga + gb;
        gsum[q] = gs;
        tw_acc[q] += gs;
        const __half h = __float2half_rn(gs);
        oh[x0 + q] = h;
        oh[KP + x0 + q] = __float2half_rn(gs - __half2float(h));
      }
      if (g) { store_row(g, g0, inv); store_row(g + K, g1, inv); }
      if (gl_) store_row(gl_, gsum, 1.f);
      if (p.gamma16) {
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          bulk_store(p.gamma16 + (size_t)t * p.ldg, oh, (uint32_t)K * 2);
          bulk_store(p.gamma16 + ((size_t)c.T + t) * p.ldg, oh + KP, (uint32_t)K * 2);
          bulk_commit();
        }
        out_par = (out_par + 1) % OB;
      }
      if (p.dyn_marg && lane == 0) {
        p.dyn_marg[2 * t] = s0 * inv;
        p.dyn_marg[2 * t + 1] = s1 * inv;
      }
      if (p.r_out && i != 0) {
        float* ro = p.r_out + (size_t)(t + 1) * 2 * K;
        store_row(ro, r0, r_scale);
        store_row(ro + K, r1, r_scale);
      }
      if (p.xr_hi && i != 0) {
        uint16_t* rh = p.xr_hi + (size_t)(t + 1) * p.ld_x;
        uint16_t* rl = p.xr_lo + (size_t)(t + 1) * p.ld_x;
        store_row_bf16(rh, rl, r0, r_scale);
        store_row_bf16(rh + K, rl + K, r1, r_scale);
      }
    } else if (t == cr.t_end && p.beta_halo) {
      float* o = p.beta_halo + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (x0 + q < K) { o[x0 + q] = b0[q] * inv; o[K + x0 + q] = b1[q] * inv; }
    }
    if (t == cr.t_begin && p.beta_end) {
      float* o = p.beta_end + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (x0 + q < K) { o[x0 + q] = b0[q] * inv; o[K + x0 + q] = b1[q] * inv; }
    }
    if (p.warm_out && t == cr.t_begin + halo_next_of(c, cr.s - 1) - 1 && (cr.s >= 1 || !c.left_exact)) {
      float* o = p.warm_out + ((int64_t)cr.s - 1) * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (x0 + q < K) { o[x0 + q] = b0[q] * inv; o[K + x0 + q] = b1[q] * inv; }
    }
  }
  if (lane == 0) bulk_wait_read<0>();
  if (p.tw_partial) {
    float* o = p.tw_partial + (size_t)cr.s * K;
#pragma unroll
    for (int q = 0; q < Q; ++q)
      if (x0 + q < K) o[x0 + q] = tw_acc[q];
  }
}

// ring depth from the shared-memory budget
template <int Q, int WT, bool FWD>
static int bulk_ring_depth(int nw, int ob, size_t budget_bytes) {
  for (int R = 8; R >= 2; --R) {
    const int f = FWD ? BulkGeo<Q, WT>::fwd_chain_floats(R, ob) : BulkGeo<Q, WT>::bwd_chain_floats(R, ob);
    if ((size_t)nw * f * sizeof(float) <= budget_bytes) return R;
  }
  return 0;
}

template <int Q, int WT, int NW, int OB>
static int launch_fwd_bulk(const FwdParams& p, int n_groups, cudaStream_t st) {
  const int R = bulk_ring_depth<Q, WT, true>(NW, OB, 216 * 1024);
  if (R == 0) return PMG_ERR_UNSUPPORTED_SHAPE;
  const size_t smem = (size_t)NW * BulkGeo<Q, WT>::fwd_chain_floats(R, OB) * sizeof(float);
  PMG_CUDA_CHECK(cudaFuncSetAttribute(fwd_bulk_kernel<Q, WT, NW, OB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fwd_bulk_kernel<Q, WT, NW, OB><<<cdiv(n_groups, NW), 32 * NW, smem, st>>>(p, R);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
template <int Q, int WT, int NW, int OB>
static int launch_bwd_bulk(const BwdParams& p, int n_groups, cudaStream_t st) {
  const int R = bulk_ring_depth<Q, WT, false>(NW, OB, 216 * 1024);
  if (R == 0) return PMG_ERR_UNSUPPORTED_SHAPE;
  const size_t smem = (size_t)NW * BulkGeo<Q, WT>::bwd_chain_floats(R, OB) * sizeof(float);
  PMG_CUDA_CHECK(cudaFuncSetAttribute(bwd_bulk_kernel<Q, WT, NW, OB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bwd_bulk_kernel<Q, WT, NW, OB><<<cdiv(n_groups, NW), 32 * NW, smem, st>>>(p, R);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

}  // namespace pmg
