// "Compact" forward / backward chain kernels: the EM-iteration fast path of the smoother.
//
// Same recursion and chain / warm-up / seam conventions as fwd_bulk_kernel / bwd_bulk_kernel
// (pmg_scan_bulk.cuh; reference decoder.py:151-187 and :200-256), specialised to what an EM iteration
// consumes (the fp16 pieces of the latent posterior and sum_t gamma) and restructured around three facts:
//
//  * the filtered jump-state message is a scalar multiple of the likelihood factor,
//      alpha_t[1,x] = a1s_t * E_t[x],   E_t[x] = exp2(s*log2e*(ll[t,x] - max_x ll[t,.])),
//    so the forward pass stores only alpha_t[0,:] plus two scalars per bin (a1s_t and the one-step
//    predictive log marginal) and the backward pass rebuilds alpha_t[1,:] from the ll row it reads anyway:
//    8K instead of 12K bytes per bin forward, 12K instead of 16K backward.  Row layout of the compact
//    buffer `ax` [T, K+4]: columns 0..K-1 = alpha_t[0,:], column K = a1s_t, column K+1 = lmr_t.
//  * all per-bin arithmetic is done on packed pairs (fma.rn.f32x2 / mul / add, sm_100), and the band
//    halo comes from the neighbouring lanes by warp shuffles (no shared-memory exchange buffer);
//  * rows leave through shared-memory staging in groups (one proxy fence per group instead of per bin)
//    and ring slots are re-armed without a proxy fence (write-after-read needs none).
//
// One warp per chain, NW chains per CTA, Toeplitz "move" kernel with half width <= WT <= Q.
// Included by pmg_scan.cu after pmg_scan_bulk.cuh.
#pragma once

namespace pmg {

struct FwdCParams {
  ScanCommon c;
  const float* carry_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  float* ax;          // [T, ldax] compact filtered posterior (see above)
  int64_t ldax;
  float* halo_state;  // [n_chain, 2, K] warmed-up message at t_begin - 1
  float* fwd_end;     // [n_chain, 2, K] true message at t_end - 1 (seam truth of the next chain), or NULL
  float* first_out;   // [2, K] true message at core_begin (sent to the left neighbour rank), or NULL
};

struct BwdCParams {
  ScanCommon c;
  const float* ax;
  int64_t ldax;
  const float* beta_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  __half* gamma16;    // [2][T][ldg] fp16 hi/lo pieces of gamma_lat
  int64_t ldg;
  float* beta_halo;
  float* beta_end;
};

__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// reciprocal and logarithm on the special-function unit (one instruction each, ~1 ulp / 2^-22): the per-bin
// normaliser only has to be positive and consistent (every step renormalises), and log c_t is added to s*max ll
// (hundreds in magnitude: one fp32 ulp of the sum is 6e-5), so the IEEE sequences (9 and 35 instructions per bin,
// the latter executed by the whole warp for lane 0's benefit) bought nothing
__device__ __forceinline__ float rcp_fast(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float log_fast(float x) {
  float y;
  asm("lg2.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y * 0.6931471805599453f;
}
__device__ __forceinline__ float2 pk(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 pk1(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 ex2_2(float2 a) { return pk(ex2_ftz(a.x), ex2_ftz(a.y)); }

// one lane of the (converged) warp, the same one every time: code under `if (elect_one())` is known to the
// compiler to run in a single thread, so bulk-copy instructions are issued straight from uniform registers
// (under `if (lane == 0)` every such instruction is wrapped in an elect/branch loop over the active lanes)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// warp-wide float max in one instruction (redux.sync.max.f32, sm_100a)
__device__ __forceinline__ float warp_max_redux(float v) {
  float r;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"(v));
  return r;
}
// two warp sums for the price of one and a half: the halves of the warp reduce different values
__device__ __forceinline__ void warp_sum2(float& a, float& b, int lane) {
  const bool hi = lane & 16;
  float keep = hi ? b : a;
  const float send = hi ? a : b;
  keep += __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) keep += __shfl_xor_sync(0xffffffffu, keep, o);
  a = __shfl_sync(0xffffffffu, keep, 0);
  b = __shfl_sync(0xffffffffu, keep, 16);
}

// out[x] = sum_{d=-WT..WT} tp[d+WT] * a[x+d] over this lane's Q = 2*QP consecutive entries; the WT entries on
// either side come from the neighbouring lanes by rotating shuffles.  Lane 31 holds only padding (zeros;
// the dispatch guarantees K <= 31*Q), so lane 0 receives the zeros that lie left of bin 0 and lane 30 the
// zeros right of bin K-1; what lane 31 itself computes lands in padding and is never used.
//
// Packed FMAs need ALIGNED register pairs.  In the window w[0 .. Q+2WT) (w[WT+i] = this lane's entry i) the aligned
// ("natural") pairs start at offsets s with s = WT (mod 2); output pair p under tap j reads the pair starting at
// 2p + j, which is natural for only half of the taps -- and the compiler re-pairs the straddling operands with
// register moves (75 per bin in the 11-tap kernel, as many as the FMAs themselves).  So the other half of the taps
// accumulates into output pairs SHIFTED by one entry, so[p] = (out[2p-1], out[2p]), whose operands start at
// 2p - 1 + j: natural again.  Every FMA operand is then a natural pair and the two partial sums meet in Q scalar adds:
//   out[2p] = nat[p].x + so[p].y,   out[2p+1] = nat[p].y + so[p+1].x.
template <int QP, int WT>
__device__ __forceinline__ void band_pk(const float2 (&a)[QP], float2 (&out)[QP], const float (&tp)[2 * WT + 1],
                                        int lane_left, int lane_right) {
  constexpr int Q = 2 * QP;
  static_assert(WT <= Q, "band half width must not exceed the lane segment");
  constexpr int NWIN = Q + 2 * WT;
  constexpr int PAR = WT & 1;              // parity of the natural pair offsets
  constexpr int S0 = PAR ? -1 : 0;         // first natural offset used (w[-1] and w[NWIN] do not exist: zeros that
                                           // only reach the discarded halves of so[0] and so[QP])
  constexpr int NP = (NWIN - S0 + 1) / 2;  // natural pairs N(S0), N(S0+2), ...
  float w[NWIN];
#pragma unroll
  for (int p = 0; p < QP; ++p) { w[WT + 2 * p] = a[p].x; w[WT + 2 * p + 1] = a[p].y; }
#pragma unroll
  for (int i = 0; i < WT; ++i) {
    w[WT - 1 - i] = __shfl_sync(0xffffffffu, w[WT + Q - 1 - i], lane_left);
    w[WT + Q + i] = __shfl_sync(0xffffffffu, w[WT + i], lane_right);
  }
  float2 nat[NP];
#pragma unroll
  for (int m = 0; m < NP; ++m) {
    const int s = S0 + 2 * m;
    if (s >= WT && s + 1 < WT + Q) nat[m] = a[(s - WT) / 2];
    else nat[m] = pk(s >= 0 ? w[s >= 0 ? s : 0] : 0.f, s + 1 < NWIN ? w[s + 1 < NWIN ? s + 1 : 0] : 0.f);
  }
  float2 so[QP + 1];
  bool so_init = false;
#pragma unroll
  for (int j = 0; j <= 2 * WT; ++j) {
    if ((j & 1) == PAR) continue;          // these taps are natural for the unshifted outputs
    const float2 t2 = pk1(tp[j]);
#pragma unroll
    for (int p = 0; p <= QP; ++p) {
      const float2 x = nat[(2 * p - 1 + j - S0) / 2];
      so[p] = so_init ? fma2(t2, x, so[p]) : mul2(t2, x);
    }
    so_init = true;
  }
  bool nat_init = false;
  float2 acc[QP];
#pragma unroll
  for (int j = 0; j <= 2 * WT; ++j) {
    if ((j & 1) != PAR) continue;
    const float2 t2 = pk1(tp[j]);
#pragma unroll
    for (int p = 0; p < QP; ++p) {
      const float2 x = nat[(2 * p + j - S0) / 2];
      acc[p] = nat_init ? fma2(t2, x, acc[p]) : mul2(t2, x);
    }
    nat_init = true;
  }
#pragma unroll
  for (int p = 0; p < QP; ++p) out[p] = pk(acc[p].x + so[p].y, acc[p].y + so[p + 1].x);
}

template <int QP>
struct CGeo {
  static constexpr int Q = 2 * QP;
  static constexpr int KP = 32 * Q;   // padded row length (floats) in shared memory
  // floats per chain: mbarriers | ring | output staging (2 groups of NB rows)
  __host__ __device__ static int fwd_floats(int R, int NB) { return round4(2 * R) + R * KP + 2 * NB * KP; }
  // ring slot = ll row | alpha0 row | 4 scalars; staging rows hold KP halves x 2 pieces = KP floats
  static constexpr int BWD_SLOT = 2 * KP + 4;
  __host__ __device__ static int bwd_floats(int R, int NB) { return round4(2 * R) + R * BWD_SLOT + 2 * NB * KP; }
};

// writes the normalised message (v0*s0, v1*s1) as a [2,K] vector
template <int QP>
__device__ __forceinline__ void store_msg(float* o, const float2 (&v0)[QP], float s0, const float2 (&v1)[QP], float s1,
                                       int x0, int K) {
#pragma unroll
  for (int p = 0; p < QP; ++p) {
    const int x = x0 + 2 * p;
    if (x < K) {       // K is even: a pair never straddles the end
      *reinterpret_cast<float2*>(o + x) = mul2(v0[p], pk1(s0));
      *reinterpret_cast<float2*>(o + K + x) = mul2(v1[p], pk1(s1));
    }
  }
}

__device__ __forceinline__ int next_event(int i, int e0, int e1, int e2, int e3) {
  int n = 0x7fffffff;
  if (e0 > i && e0 < n) n = e0;
  if (e1 > i && e1 < n) n = e1;
  if (e2 > i && e2 < n) n = e2;
  if (e3 > i && e3 < n) n = e3;
  return n;
}

// ============================================================================
// forward
// ============================================================================
template <int QP, int WT, int NW, int NB>
__global__ void __launch_bounds__(32 * NW, 1) fwd_c_kernel(const FwdCParams p, const int R) {
  using G = CGeo<QP>;
  constexpr int Q = G::Q, KP = G::KP;
  extern __shared__ __align__(16) float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, NW)) return;
  const int K = c.tr.K, W = c.tr.W;
  const int grp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int lane_left = (lane + 31) & 31, lane_right = (lane + 1) & 31;
  const int x0 = lane * Q;

  float* base = smem + (size_t)grp * G::fwd_floats(R, NB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base);
  float* ring = base + round4(2 * R);            // R rows of KP floats; columns >= K stay -inf
  float* outb = ring + (size_t)R * KP;           // 2 groups x NB rows x KP floats
  for (int i = lane; i < R * KP; i += 32) ring[i] = -INFINITY;
  for (int i = lane; i < 2 * NB * KP; i += 32) outb[i] = 0.f;
  if (lane == 0) {
    for (int s = 0; s < R; ++s) tc::mbar_init(&bars[s], 1);
    tc::fence_barrier_init();
  }
  fence_proxy_async();
  __syncthreads();

  ChainRange cr;
  if (!chain_range<NW>(c, grp, cr)) return;

  // taps carry M00: prior move message = M00 * band(iz * u), u = v0 + (M10/M00) v1, v1 = p1 * Lc
  const float M00 = c.tr.M00, M01 = c.tr.M01, M11 = c.tr.M11;
  const float cM = c.tr.M10 / M00;
  float tp[2 * WT + 1];
#pragma unroll
  for (int j = 0; j <= 2 * WT; ++j) {
    const int d = j >= WT ? j - WT : WT - j;
    tp[j] = d <= W ? M00 * __ldg(c.tr.taps + d) : 0.f;
  }
  float2 iz2[QP];
#pragma unroll
  for (int q = 0; q < QP; ++q) {
    const int x = x0 + 2 * q;
    iz2[q] = x < K ? pk(__ldg(c.tr.inv_z + x), __ldg(c.tr.inv_z + x + 1)) : pk1(0.f);
  }
  const float invK = 1.f / (float)K;
  const float sc2 = c.scale * kLog2e;

  // ---- initial carry
  int64_t t0;
  const float* src = fwd_start<false>(c, cr, p, t0, K);   // no alpha to restart from
  // u = v0 + cM * v1 (unnormalised), S0 = sum v0, S1 = sum v1, inv_prev = 1 / (S0 + S1)
  float2 u[QP];
  float S0 = 0.f, S1 = 0.f;
  {
    float2 a0[QP], a1[QP];
#pragma unroll
    for (int q = 0; q < QP; ++q) {
      const int x = x0 + 2 * q;
      const bool ok = x < K;
      a0[q] = ok ? (src ? pk(src[x], src[x + 1]) : pk1(0.5f * invK)) : pk1(0.f);
      a1[q] = ok ? (src ? pk(src[K + x], src[K + x + 1]) : pk1(0.5f * invK)) : pk1(0.f);
      S0 += a0[q].x + a0[q].y;
      S1 += a1[q].x + a1[q].y;
    }
    S0 = warp_sum(S0); S1 = warp_sum(S1);
    if (!(S0 + S1 > 0.f) || !(S0 + S1 < 3.0e38f)) {      // unusable initial message: uniform
#pragma unroll
      for (int q = 0; q < QP; ++q) { a0[q] = (x0 + 2 * q < K) ? pk1(0.5f * invK) : pk1(0.f); a1[q] = a0[q]; }
      S0 = 0.5f; S1 = 0.5f;
    }
#pragma unroll
    for (int q = 0; q < QP; ++q) u[q] = fma2(pk1(cM), a1[q], a0[q]);
  }
  float inv_prev = 1.f / (S0 + S1);

  // ---- step indices of the rare events (all relative to t0)
  const int n_steps = (int)(cr.t_end - t0);
  const int i_begin = (int)(cr.t_begin - t0);                    // first bin whose row is stored
  const int e_halo = p.halo_state ? i_begin - 1 : -1;            // warmed-up message in front of the chain
  const int e_warm = (p.warm_out && (cr.s + 1 < c.n_chain || !c.right_exact)) ? (int)(cr.t_end - halo_next_of(c, cr.s + 1) - 1 - t0) : -1;
  const int e_end = p.fwd_end ? n_steps - 1 : -1;
  const int e_first = (p.first_out && cr.t_begin == c.core_begin) ? i_begin : -1;
  int evt = next_event(-1, e_halo, e_warm, e_end, e_first);

  // ---- fill the input ring
  const uint32_t row_bytes = (uint32_t)K * 4;
  const float* ll_next = c.ll + (size_t)t0 * c.ldll;             // row the next refill loads
  if (elect_one()) {
    for (int j = 0; j < R && j < n_steps; ++j) {
      tc::mbar_arrive_expect_tx(&bars[j], row_bytes);
      bulk_load(ring + (size_t)j * KP, ll_next + (size_t)j * c.ldll, row_bytes, &bars[j]);
    }
  }
  ll_next += (size_t)R * c.ldll;
  float* ax_row = p.ax + (size_t)cr.t_begin * p.ldax;            // row of the next stored bin

  int slot = 0, og = 0, orow = 0;
  uint32_t ring_phase = 0;
  float* ax_group = ax_row;                                      // first row of the group being staged
  for (int i = 0; i < n_steps; ++i) {
    if (orow == 0 && i >= i_begin) {             // a new staging group starts: its buffer must have been read out
      if (elect_one()) bulk_wait_read<1>();
      __syncwarp();
    }
    tc::mbar_wait(&bars[slot], ring_phase);
    float2 Lc[QP];
    float m = -INFINITY;
    {
      const float* row = ring + (size_t)slot * KP + x0;
#pragma unroll
      for (int q = 0; q < QP; ++q) {
        Lc[q] = *reinterpret_cast<const float2*>(row + 2 * q);
        m = fmaxf(m, fmaxf(Lc[q].x, Lc[q].y));
      }
    }
    // carried message -> banded operator (the loop-carried chain)
    float2 a[QP], pr0[QP];
#pragma unroll
    for (int q = 0; q < QP; ++q) a[q] = mul2(iz2[q], u[q]);
    band_pk<QP, WT>(a, pr0, tp, lane_left, lane_right);
    // every lane holds its part of ring[slot] in registers: refill the slot R steps ahead
    __syncwarp();
    if (i + R < n_steps) {
      if (elect_one()) {
        tc::mbar_arrive_expect_tx(&bars[slot], row_bytes);
        bulk_load(ring + (size_t)slot * KP, ll_next, row_bytes, &bars[slot]);
      }
    }
    ll_next += c.ldll;
    if (++slot == R) { slot = 0; ring_phase ^= 1; }

    // likelihood factor (previous normaliser folded in), new message, normaliser
    m = warp_max_redux(m);
    const float2 s2 = pk1(sc2), nm2 = pk1(-m * sc2), ip2 = pk1(inv_prev);
    const float p1 = (M01 * S0 + M11 * S1) * invK;
    float2 v0[QP];
    float2 s0 = pk1(0.f), sL = pk1(0.f);
#pragma unroll
    for (int q = 0; q < QP; ++q) {
      Lc[q] = mul2(ex2_2(fma2(Lc[q], s2, nm2)), ip2);          // pads: exp2(-inf) = 0
      v0[q] = mul2(pr0[q], Lc[q]);
      s0 = add2(s0, v0[q]);
      sL = add2(sL, Lc[q]);
    }
    S0 = s0.x + s0.y;
    S1 = sL.x + sL.y;
    warp_sum2(S0, S1, lane);
    S1 *= p1;
    const float cn = S0 + S1;                    // c_t = sum of prior x likelihood
    const float inv = rcp_fast(cn);

    if (i >= i_begin) {
      float* ob = outb + (size_t)(og * NB + orow) * KP + x0;
      const float2 i2 = pk1(inv);
#pragma unroll
      for (int q = 0; q < QP; ++q) *reinterpret_cast<float2*>(ob + 2 * q) = mul2(v0[q], i2);
      if (lane == 0) *reinterpret_cast<float2*>(ax_row + K) = pk(p1 * inv_prev * inv, log_fast(cn) + c.scale * m);
      ax_row += p.ldax;
      ++orow;
      if (orow == NB || i == n_steps - 1) {
        fence_proxy_async();
        __syncwarp();
        if (elect_one()) {
          for (int r = 0; r < orow; ++r)
            bulk_store(ax_group + (size_t)r * p.ldax, outb + (size_t)(og * NB + r) * KP, row_bytes);
          bulk_commit();
        }
        ax_group = ax_row;
        orow = 0;
        og ^= 1;
      }
    }
    if (i == evt) {                              // rare: seam / warm-start messages (normalised [2,K] vectors)
      const float s1 = p1 * inv;
      if (i == e_halo) store_msg<QP>(p.halo_state + (size_t)cr.s * 2 * K, v0, inv, Lc, s1, x0, K);
      if (i == e_warm) store_msg<QP>(p.warm_out + (size_t)(cr.s + 1) * 2 * K, v0, inv, Lc, s1, x0, K);
      if (i == e_end) store_msg<QP>(p.fwd_end + (size_t)cr.s * 2 * K, v0, inv, Lc, s1, x0, K);
      if (i == e_first) store_msg<QP>(p.first_out, v0, inv, Lc, s1, x0, K);
      evt = next_event(i, e_halo, e_warm, e_end, e_first);
    }
    const float2 c1 = pk1(cM * p1);
#pragma unroll
    for (int q = 0; q < QP; ++q) u[q] = fma2(c1, Lc[q], v0[q]);
    inv_prev = inv;
  }
  __syncwarp();
  if (elect_one()) bulk_wait_read<0>();
}

// ============================================================================
// backward
// ============================================================================
template <int QP, int WT, int NW, int NB>
__global__ void __launch_bounds__(32 * NW, 1) bwd_c_kernel(const BwdCParams p, const int R) {
  using G = CGeo<QP>;
  constexpr int Q = G::Q, KP = G::KP;
  constexpr int SLOT = G::BWD_SLOT;
  extern __shared__ __align__(16) float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, NW)) return;
  const int K = c.tr.K, W = c.tr.W;
  const int grp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int lane_left = (lane + 31) & 31, lane_right = (lane + 1) & 31;
  const int x0 = lane * Q;

  float* base = smem + (size_t)grp * G::bwd_floats(R, NB);
  uint64_t* bars = reinterpret_cast<uint64_t*>(base);
  float* ring = base + round4(2 * R);            // slot: [ll KP | alpha0 KP | a1s, lmr, -, -]
  __half* outh = reinterpret_cast<__half*>(ring + (size_t)R * SLOT);   // 2 groups x NB rows x (hi KP | lo KP) halves
  for (int i = lane; i < R * SLOT; i += 32) ring[i] = ((i % SLOT) < KP) ? -INFINITY : 0.f;
  for (int i = lane; i < 2 * NB * KP; i += 32) reinterpret_cast<float*>(outh)[i] = 0.f;
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
  // beta_t[d,x] = M[d,0] * band(r0)[x] / z[x] + M[d,1] * w1
  float2 iz2[QP];
#pragma unroll
  for (int q = 0; q < QP; ++q) {
    const int x = x0 + 2 * q;
    iz2[q] = x < K ? pk(__ldg(c.tr.inv_z + x), __ldg(c.tr.inv_z + x + 1)) : pk1(0.f);
  }
  const float2 M00_2 = pk1(c.tr.M00), M10_2 = pk1(c.tr.M10);
  const float M01 = c.tr.M01, M11 = c.tr.M11;
  const float invK = 1.f / (float)K;
  const float sc2 = c.scale * kLog2e;

  int64_t t_hi;
  const float* init = bwd_start<true>(c, cr, p, t_hi, K);

  // carried: unnormalised beta (b0, b1) of the bin handled last, its likelihood factor with the normaliser
  // folded in (Lb), the unnormalised jump-state sum RLu = sum_x E*b1 and the normaliser inv_prev
  float2 b0[QP], b1[QP], Lb[QP];
  float inv_prev = 1.f, RLu = 0.f;
#pragma unroll
  for (int q = 0; q < QP; ++q) {
    const int x = x0 + 2 * q;
    const bool ok = x < K;
    b0[q] = ok ? (init ? pk(init[x], init[x + 1]) : pk1(1.f)) : pk1(0.f);
    b1[q] = ok ? (init ? pk(init[K + x], init[K + x + 1]) : pk1(1.f)) : pk1(0.f);
    Lb[q] = pk1(0.f);
  }
  {
    float sb = 0.f;
#pragma unroll
    for (int q = 0; q < QP; ++q) sb += b0[q].x + b0[q].y + b1[q].x + b1[q].y;
    sb = warp_sum(sb);
    if (!(sb > 0.f) || !(sb < 3.0e38f)) {        // unusable initial message: all ones
#pragma unroll
      for (int q = 0; q < QP; ++q) { b0[q] = (x0 + 2 * q < K) ? pk1(1.f) : pk1(0.f); b1[q] = b0[q]; }
    }
  }

  // ---- step indices (step i handles bin t_hi - i); the filtered posterior is needed for bins <= t_end
  const int n_steps = (int)(t_hi - cr.t_begin + 1);
  const int i_alpha = (int)(t_hi - cr.t_end);                    // first step that uses alpha (may be < 0)
  const int i_core = (int)(t_hi - (cr.t_end - 1));               // first step of the chain's own bins
  const int e_halo = (p.beta_halo && i_alpha >= 0) ? i_alpha : -1;          // t == t_end
  const int e_end = p.beta_end ? n_steps - 1 : -1;                          // t == t_begin
  const int e_warm = (p.warm_out && (cr.s >= 1 || !c.left_exact)) ? (int)(t_hi - (cr.t_begin + halo_next_of(c, cr.s - 1) - 1)) : -1;
  int evt = next_event(-1, e_halo, e_end, e_warm, -1);

  const uint32_t row_bytes = (uint32_t)K * 4;
  const float* ll_next = c.ll + (size_t)t_hi * c.ldll;
  const float* ax_next = p.ax + (size_t)t_hi * p.ldax;
  auto issue = [&](int s, int step) {
    const bool need_a = step >= i_alpha;
    tc::mbar_arrive_expect_tx(&bars[s], need_a ? 2 * row_bytes + 16 : row_bytes);
    float* dst = ring + (size_t)s * SLOT;
    bulk_load(dst, ll_next, row_bytes, &bars[s]);
    if (need_a) {
      bulk_load(dst + KP, ax_next, row_bytes, &bars[s]);
      bulk_load(dst + 2 * KP, ax_next + K, 16, &bars[s]);
    }
  };
  for (int j = 0; j < R; ++j) {
    if (j < n_steps) {
      if (elect_one()) issue(j, j);
    }
    ll_next -= c.ldll;
    ax_next -= p.ldax;
  }

  // output groups are aligned to t_begin: bin t goes to row (t - t_begin) % NB of its group and the group is
  // flushed when row 0 has been written (bins are visited in descending order)
  int slot = 0, og = 0;
  uint32_t ring_phase = 0;
  int r_out = (int)((cr.t_end - 1 - cr.t_begin) % NB);           // staging row of the next core bin
  int n_rows = r_out + 1;                                        // rows of the group being staged
  __half* g_row = p.gamma16 + (size_t)(cr.t_end - 1) * p.ldg;    // global row (hi piece) of the next core bin
  const size_t piece = (size_t)c.T * p.ldg;
  for (int i = 0; i < n_steps; ++i) {
    const bool core = i >= i_core;
    if (core && r_out == n_rows - 1) {           // a new staging group starts
      if (elect_one()) bulk_wait_read<1>();
      __syncwarp();
    }
    tc::mbar_wait(&bars[slot], ring_phase);
    const float* row = ring + (size_t)slot * SLOT + x0;

    // ---- unnormalised beta_t (carried chain: b -> band -> b); step 0 uses the initial message as is
    if (i > 0) {
      float2 r0[QP], w0[QP];
#pragma unroll
      for (int q = 0; q < QP; ++q) r0[q] = mul2(Lb[q], b0[q]);      // Lb carries 1/normaliser; pads are 0
      band_pk<QP, WT>(r0, w0, tp, lane_left, lane_right);
      const float w1 = RLu * inv_prev * invK;
      const float2 c0 = pk1(M01 * w1), c1 = pk1(M11 * w1);
#pragma unroll
      for (int q = 0; q < QP; ++q) {             // pad entries are finite garbage; E = 0 and alpha = 0 there
        const float2 zw = mul2(iz2[q], w0[q]);
        b0[q] = fma2(M00_2, zw, c0);
        b1[q] = fma2(M10_2, zw, c1);
      }
    }

    // ---- likelihood factor of this bin, normaliser, posterior
    float2 E[QP];
    float m = -INFINITY;
#pragma unroll
    for (int q = 0; q < QP; ++q) {
      E[q] = *reinterpret_cast<const float2*>(row + 2 * q);
      m = fmaxf(m, fmaxf(E[q].x, E[q].y));
    }
    m = warp_max_redux(m);
    const float2 s2v = pk1(sc2), nm2 = pk1(-m * sc2);
    float2 g0[QP], e[QP];
    float2 s0 = pk1(0.f), s2 = pk1(0.f);
    float a1s = 1.f;
    if (i >= i_alpha) {
      a1s = row[2 * KP - x0];                    // ring[slot][2*KP]: broadcast read
#pragma unroll
      for (int q = 0; q < QP; ++q) {
        E[q] = ex2_2(fma2(E[q], s2v, nm2));
        g0[q] = mul2(*reinterpret_cast<const float2*>(row + KP + 2 * q), b0[q]);
        e[q] = mul2(E[q], b1[q]);
        s0 = add2(s0, g0[q]);
        s2 = add2(s2, e[q]);
      }
    } else {
      // warm-up beyond the chain's own bins: any positive normaliser works; use sum_x E*(b0+b1)
#pragma unroll
      for (int q = 0; q < QP; ++q) {
        E[q] = ex2_2(fma2(E[q], s2v, nm2));
        g0[q] = mul2(E[q], b0[q]);
        e[q] = mul2(E[q], b1[q]);
        s0 = add2(s0, g0[q]);
        s2 = add2(s2, e[q]);
      }
    }
    // all lanes are done with ring[slot]: refill it R steps ahead
    __syncwarp();
    if (i + R < n_steps) {
      if (elect_one()) issue(slot, i + R);
    }
    ll_next -= c.ldll;
    ax_next -= p.ldax;
    if (++slot == R) { slot = 0; ring_phase ^= 1; }

    float S0 = s0.x + s0.y, S2 = s2.x + s2.y;
    warp_sum2(S0, S2, lane);
    const float inv = rcp_fast(S0 + a1s * S2);
    const float2 i2 = pk1(inv);

    if (core) {
      __half2* hi = reinterpret_cast<__half2*>(outh + (size_t)(og * NB + r_out) * 2 * KP) + lane * QP;
      __half2* lo = hi + KP / 2;
      const float2 a2 = pk1(a1s);
#pragma unroll
      for (int q = 0; q < QP; ++q) {
        const float2 gl = mul2(fma2(a2, e[q], g0[q]), i2);     // gamma_lat = (alpha0 b0 + alpha1 b1) / z
        const __half2 h = __floats2half2_rn(gl.x, gl.y);
        const float2 hf = __half22float2(h);
        hi[q] = h;
        lo[q] = __floats2half2_rn(gl.x - hf.x, gl.y - hf.y);
      }
      if (r_out == 0) {
        fence_proxy_async();
        __syncwarp();
        if (elect_one()) {
          for (int rr = 0; rr < n_rows; ++rr) {
            const __half* srow = outh + (size_t)(og * NB + rr) * 2 * KP;
            bulk_store(g_row + (size_t)rr * p.ldg, srow, (uint32_t)K * 2);
            bulk_store(g_row + piece + (size_t)rr * p.ldg, srow + KP, (uint32_t)K * 2);
          }
          bulk_commit();
        }
        og ^= 1;
        r_out = NB - 1;
        n_rows = NB;
      } else {
        --r_out;
      }
      g_row -= p.ldg;
    }
    if (i == evt) {                              // rare: seam / warm-start messages (normalised beta)
      if (i == e_halo) store_msg<QP>(p.beta_halo + (size_t)cr.s * 2 * K, b0, inv, b1, inv, x0, K);
      if (i == e_end) store_msg<QP>(p.beta_end + (size_t)cr.s * 2 * K, b0, inv, b1, inv, x0, K);
      if (i == e_warm) store_msg<QP>(p.warm_out + ((int64_t)cr.s - 1) * 2 * K, b0, inv, b1, inv, x0, K);
      evt = next_event(i, e_halo, e_end, e_warm, -1);
    }
#pragma unroll
    for (int q = 0; q < QP; ++q) Lb[q] = mul2(E[q], i2);
    RLu = S2;
    inv_prev = inv;
  }
  __syncwarp();
  if (elect_one()) bulk_wait_read<0>();
}

// ---- host side ---------------------------------------------------------------------------
constexpr size_t kCompactSmemBudget = 224 * 1024;

template <int QP, bool FWD>
static int compact_ring_depth(int nw, int nb) {
  for (int R = 8; R >= 3; --R) {
    const int f = FWD ? CGeo<QP>::fwd_floats(R, nb) : CGeo<QP>::bwd_floats(R, nb);
    if ((size_t)nw * f * sizeof(float) <= kCompactSmemBudget) return R;
  }
  return 0;
}

template <int QP, int WT, int NW>
static int launch_fwd_c(const FwdCParams& p, int n_groups, cudaStream_t st) {
  constexpr int NB = NW > 8 ? 2 : 4;
  const int R = compact_ring_depth<QP, true>(NW, NB);
  if (R == 0) return PMG_ERR_UNSUPPORTED_SHAPE;
  const size_t smem = (size_t)NW * CGeo<QP>::fwd_floats(R, NB) * sizeof(float);
  PMG_CUDA_CHECK(cudaFuncSetAttribute(fwd_c_kernel<QP, WT, NW, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fwd_c_kernel<QP, WT, NW, NB><<<cdiv(n_groups, NW), 32 * NW, smem, st>>>(p, R);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
template <int QP, int WT, int NW>
static int launch_bwd_c(const BwdCParams& p, int n_groups, cudaStream_t st) {
  constexpr int NB = 2;
  const int R = compact_ring_depth<QP, false>(NW, NB);
  if (R == 0) return PMG_ERR_UNSUPPORTED_SHAPE;
  const size_t smem = (size_t)NW * CGeo<QP>::bwd_floats(R, NB) * sizeof(float);
  PMG_CUDA_CHECK(cudaFuncSetAttribute(bwd_c_kernel<QP, WT, NW, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bwd_c_kernel<QP, WT, NW, NB><<<cdiv(n_groups, NW), 32 * NW, smem, st>>>(p, R);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

// (pairs per lane, band capacity) for a supported shape, or QP = 0
static void compact_geometry(const pmg_transition* tr, int& QP, int& WT) {
  QP = 0; WT = 0;
  if (!tr || tr->kind != 0 || tr->K < 8 || (tr->K & 7) || tr->W > 10) return;
  if (!(tr->M[0] > 0.f)) return;                 // the forward kernel folds M00 into the taps
  const int K = tr->K;                           // lane 31 must hold only padding: K <= 31 * 2 * QP
  if (tr->W <= 5) {
    WT = 5;
    QP = K <= 31 * 8 ? 4 : K <= 31 * 14 ? 7 : K <= 31 * 16 ? 8 : 0;
  } else {
    WT = 10;
    QP = K <= 31 * 14 ? 7 : K <= 31 * 16 ? 8 : 0;
  }
}

template <bool FWD, typename P>
static int dispatch_compact(const P& p, const pmg_transition* tr, int n_groups, cudaStream_t st) {
  int QP, WT;
  compact_geometry(tr, QP, WT);
  // 12 chains per CTA (3 warps per scheduler) when the plan has more chains than 8 per SM can hold at once
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const bool wide = n_groups > 8 * sms;
#define PMG_CC(QPv, WTv, NWv)                                                   \
  if (QP == QPv && WT == WTv) {                                                 \
    if constexpr (FWD) return launch_fwd_c<QPv, WTv, NWv>(p, n_groups, st);     \
    else return launch_bwd_c<QPv, WTv, NWv>(p, n_groups, st);                   \
  }
  if (wide) { PMG_CC(7, 5, 12) PMG_CC(8, 5, 12) }
  PMG_CC(4, 5, 8) PMG_CC(7, 5, 8) PMG_CC(8, 5, 8) PMG_CC(7, 10, 8) PMG_CC(8, 10, 8)
#undef PMG_CC
  return PMG_ERR_UNSUPPORTED_SHAPE;
}

}  // namespace pmg

extern "C" int pmg_scan_compact_supported(const pmg_transition* tr, float likelihood_scale) {
  int QP, WT;
  pmg::compact_geometry(tr, QP, WT);
  return QP > 0 && likelihood_scale > 0.f;
}

extern "C" int pmg_forward_compact(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                                   const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                                   float* ax, int64_t ldax, float* halo_state, float* fwd_end, float* first_out,
                                   int mode, const int* chain_ids, int n_ids, pmg_stream_t stream) {
  pmg::FwdCParams p;
  int rc = pmg::fill_common(p.c, plan, tr, ll, ldll, mode, chain_ids, n_ids, true);
  if (rc) return rc;
  if (!ax || ldax < tr->K + 4 || (ldax & 3) || (ldll & 3)) return PMG_ERR_BAD_ARG;
  if (!pmg_scan_compact_supported(tr, plan->likelihood_scale)) return PMG_ERR_UNSUPPORTED_SHAPE;
  if (((uintptr_t)ll | (uintptr_t)ax) & 15) return PMG_ERR_ALIGNMENT;
  if (mode != 0 && !warm_in) return PMG_ERR_BAD_ARG;      // relays restart from a snapshot of the carry
  p.carry_in = carry_in; p.warm_in = warm_in; p.warm_stride = warm_stride; p.warm_out = warm_out;
  p.ax = ax; p.ldax = ldax; p.halo_state = halo_state; p.fwd_end = fwd_end; p.first_out = first_out;
  const int n_groups = mode == 1 ? n_ids : plan->n_chain;
  return pmg::dispatch_compact<true>(p, tr, n_groups, (cudaStream_t)stream);
}

extern "C" int pmg_backward_compact(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                                    const float* ax, int64_t ldax, const float* beta_in, const float* warm_in,
                                    int64_t warm_stride, float* warm_out, void* gamma16, int64_t ldg,
                                    float* beta_halo, float* beta_end, int mode,
                                    const int* chain_ids, int n_ids, pmg_stream_t stream) {
  pmg::BwdCParams p;
  int rc = pmg::fill_common(p.c, plan, tr, ll, ldll, mode, chain_ids, n_ids, false);
  if (rc) return rc;
  if (!ax || ldax < tr->K + 4 || (ldax & 3) || (ldll & 3)) return PMG_ERR_BAD_ARG;
  if (!gamma16 || ldg < tr->K || (ldg & 7)) return PMG_ERR_BAD_ARG;
  if (!pmg_scan_compact_supported(tr, plan->likelihood_scale)) return PMG_ERR_UNSUPPORTED_SHAPE;
  if (((uintptr_t)ll | (uintptr_t)ax | (uintptr_t)gamma16) & 15) return PMG_ERR_ALIGNMENT;
  if (mode != 0 && !beta_end && !warm_in) return PMG_ERR_BAD_ARG;
  p.ax = ax; p.ldax = ldax; p.beta_in = beta_in; p.warm_in = warm_in; p.warm_stride = warm_stride;
  p.warm_out = warm_out; p.gamma16 = (__half*)gamma16; p.ldg = ldg;
  p.beta_halo = beta_halo; p.beta_end = beta_end;
  const int n_groups = mode == 1 ? n_ids : plan->n_chain;
  return pmg::dispatch_compact<false>(p, tr, n_groups, (cudaStream_t)stream);
}
