// Forward filter / backward smoother of the joint latent x {move, jump} HMM in
// linear space, parallel in time over contiguous chunks ("chains").
//
// Replaces reference poor_man_gplvm/decoder.py:151-198 (filter_one_step /
// filter_all_step) and :200-332 (smooth_one_step / smooth_all_step /
// smooth_all_step_combined_ma_chunk); algebra in SURVEY.md Appendix A.
//
// A chain is owned by a group of 32*WPC threads; each thread keeps Q latent
// bins of the carried message in registers.  Per time step the "move" part of
// the transition (a banded K x K operator, Toeplitz for the default RBF kernel)
// is applied through a shared-memory exchange of the message, the rank-1 "jump"
// part through a group reduction that is fused with the normaliser.
#include <cuda_fp16.h>

#include "pmg_chain.cuh"

namespace pmg {

struct FwdParams {
  ScanCommon c;
  const float* carry_in;
  const float* warm_in;     // initial message of approximate (warm-up) starts: [2K] (stride 0) or per chain
  int64_t warm_stride;
  float* warm_out;          // [n_chain][2K]: message at the next chain's warm-up start (for the next pass)
  float* alpha;
  float* lmr;
  float* halo_state;
};

struct BwdParams {
  ScanCommon c;
  const float* alpha;
  const float* beta_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  float* gamma;
  float* gamma_lat;
  __half* gamma16;       // [2][T][ldg]: fp16 hi/lo pieces of gamma_lat for the tensor-core statistics GEMM
  int64_t ldg;
  float* dyn_marg;
  float* r_out;
  float* tw_partial;
  float* beta_halo;
  float* beta_end;
  // operands of the transition-count GEMM as bf16 hi/lo pieces, written in place of the fp32 r (bulk kernel only):
  // row t of xa_* = alpha_t [2K], row t+1 of xr_* = r_{t+1} / z_t [2K]; leading dimension ld_x (elements)
  uint16_t* xa_hi;
  uint16_t* xa_lo;
  uint16_t* xr_hi;
  uint16_t* xr_lo;
  int64_t ld_x;
};

template <int Q, int WPC, int WT>
struct Geo {
  static constexpr int G = 32 * WPC;       // threads per chain
  static constexpr int CPC = 8 / WPC;      // chains per 256-thread CTA
  static constexpr bool REG = WT > 0;      // register-window Toeplitz path
  static constexpr int STR = (Q % 2 == 0) ? Q + 1 : Q;   // odd chunk stride: conflict-free
  static constexpr int PADC = REG ? (WT + Q - 1) / Q : 0;
  static constexpr int KP = G * Q;
  __host__ __device__ static int buf_floats(int W) {
    return REG ? (G + 2 * PADC) * STR : (KP + 2 * W);
  }
  // dynamic smem: per chain 2 exchange buffers + 2 reduction scratch rows; taps for the generic path
  __host__ __device__ static size_t smem_bytes(int W) {
    return sizeof(float) * ((size_t)CPC * (2 * buf_floats(W) + 2 * WPC * 4) + (REG ? 0 : (W + 1)));
  }
};

// ---- banded "move" operator ------------------------------------------------
// in[q]  : this thread's Q entries of the input vector (already scaled for the Toeplitz forward case)
// out[q] : sum over the band.  `band` = band_fwd (forward) or band_bwd (backward) for kind 1.
template <int Q, int WPC, int WT>
__device__ __forceinline__ void band_apply(const float (&in)[Q], float (&out)[Q], float* buf, int gl,
                                           const float (&tp)[2 * WT + 1], const float* tapsS,
                                           const float* band, int kind, int W, int K, int bar_id) {
  using Ge = Geo<Q, WPC, WT>;
  if constexpr (Ge::REG) {
#pragma unroll
    for (int q = 0; q < Q; ++q) buf[(gl + Ge::PADC) * Ge::STR + q] = in[q];
    group_sync<WPC>(bar_id);
    float win[Q + 2 * WT];
#pragma unroll
    for (int i = 0; i < Q + 2 * WT; ++i) {
      const int e = i - WT;
      const int co = (e >= 0) ? (e / Q) : -((-e + Q - 1) / Q);
      win[i] = buf[(gl + Ge::PADC + co) * Ge::STR + (e - co * Q)];
    }
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      float acc = 0.f;
#pragma unroll
      for (int j = 0; j <= 2 * WT; ++j) acc = fmaf(tp[j], win[q + j], acc);
      out[q] = acc;
    }
  } else {
#pragma unroll
    for (int q = 0; q < Q; ++q) buf[W + gl + Ge::G * q] = in[q];
    group_sync<WPC>(bar_id);
#pragma unroll
    for (int q = 0; q < Q; ++q) out[q] = 0.f;
    if (kind == 0) {
      for (int j = 0; j <= 2 * W; ++j) {
        const float w = tapsS[j >= W ? j - W : W - j];
#pragma unroll
        for (int q = 0; q < Q; ++q) out[q] = fmaf(w, buf[gl + Ge::G * q + j], out[q]);
      }
    } else {
      for (int j = 0; j <= 2 * W; ++j) {
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          const int x = gl + Ge::G * q;
          const float w = (x < K) ? __ldg(band + (size_t)j * K + x) : 0.f;
          out[q] = fmaf(w, buf[x + j], out[q]);
        }
      }
    }
  }
}

template <int Q, int WPC, int WT>
__device__ __forceinline__ int own_x(int gl, int q) {
  return Geo<Q, WPC, WT>::REG ? gl * Q + q : gl + Geo<Q, WPC, WT>::G * q;
}

// ============================================================================
// forward
// ============================================================================
template <int Q, int WPC, int WT>
__global__ void __launch_bounds__(256, 1) fwd_kernel(const FwdParams p) {
  using Ge = Geo<Q, WPC, WT>;
  extern __shared__ float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, Geo<Q, WPC, WT>::CPC)) return;
  const int K = c.tr.K, W = c.tr.W, kind = c.tr.kind;
  const int grp = threadIdx.x / Ge::G;
  const int gl = threadIdx.x % Ge::G;
  const int lane = threadIdx.x & 31;
  const int wig = gl >> 5;
  const int bar_id = 1 + grp;

  const int bf = Ge::buf_floats(W);
  float* buf0 = smem + (size_t)grp * (2 * bf + 2 * WPC * 4);
  float* red = buf0 + 2 * bf;
  float* tapsS = smem + (size_t)Ge::CPC * (2 * bf + 2 * WPC * 4);
  if (!Ge::REG) {
    if (kind == 0)
      for (int i = threadIdx.x; i <= W; i += blockDim.x) tapsS[i] = c.tr.taps[i];
  }
  for (int i = threadIdx.x; i < Ge::CPC * (2 * bf + 2 * WPC * 4); i += blockDim.x) smem[i] = 0.f;
  __syncthreads();

  ChainRange cr;
  if (!chain_range<Ge::CPC>(c, grp, cr)) return;

  float tp[2 * WT + 1];
  if constexpr (Ge::REG) {
#pragma unroll
    for (int j = 0; j <= 2 * WT; ++j) {
      const int d = j >= WT ? j - WT : WT - j;
      tp[j] = d <= W ? __ldg(c.tr.taps + d) : 0.f;
    }
  }
  float invz[Q];
  bool valid[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int x = own_x<Q, WPC, WT>(gl, q);
    valid[q] = x < K;
    invz[q] = (kind == 0 && valid[q]) ? __ldg(c.tr.inv_z + x) : 1.f;
  }
  const float M00 = c.tr.M00, M01 = c.tr.M01, M10 = c.tr.M10, M11 = c.tr.M11;
  const float invK = 1.f / (float)K;
  const float scale = c.scale;
  int red_par = 0;

  // ---- initial carry
  int64_t t0;
  float al0[Q], al1[Q];
  const float* src = fwd_start<true>(c, cr, p, t0, K);
  float p1;
  if (src) {
    float s2[2] = {0.f, 0.f};
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int x = own_x<Q, WPC, WT>(gl, q);
      al0[q] = valid[q] ? src[x] : 0.f;
      al1[q] = valid[q] ? src[K + x] : 0.f;
      s2[0] += al0[q];
      s2[1] += al1[q];
    }
    group_sum<WPC, 2>(s2, red, red_par, wig, lane, bar_id);
    const float tot = s2[0] + s2[1];
    if (tot > 0.f && tot < 3.0e38f) {
      const float inv = 1.f / tot;
#pragma unroll
      for (int q = 0; q < Q; ++q) { al0[q] *= inv; al1[q] *= inv; }
      p1 = (M01 * s2[0] + M11 * s2[1]) * inv * invK;
    } else {   // unusable initial message: uniform
      const float u = 0.5f * invK;
#pragma unroll
      for (int q = 0; q < Q; ++q) { al0[q] = valid[q] ? u : 0.f; al1[q] = al0[q]; }
      p1 = (M01 * 0.5f + M11 * 0.5f) * invK;
    }
  } else {
    const float u = 0.5f * invK;
#pragma unroll
    for (int q = 0; q < Q; ++q) { al0[q] = valid[q] ? u : 0.f; al1[q] = al0[q]; }
    p1 = (M01 * 0.5f + M11 * 0.5f) * invK;
  }

  // ---- prefetch ll[t0]
  float lln[Q];
  {
    const float* row = c.ll + (size_t)t0 * c.ldll;
#pragma unroll
    for (int q = 0; q < Q; ++q) lln[q] = valid[q] ? __ldg(row + own_x<Q, WPC, WT>(gl, q)) : -INFINITY;
  }

  int par = 0;
  for (int64_t t = t0; t < cr.t_end; ++t) {
    float llc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) llc[q] = lln[q];
    if (t + 1 < cr.t_end) {
      const float* row = c.ll + (size_t)(t + 1) * c.ldll;
#pragma unroll
      for (int q = 0; q < Q; ++q) lln[q] = valid[q] ? __ldg(row + own_x<Q, WPC, WT>(gl, q)) : -INFINITY;
    }
    // likelihood factor L_t = exp(s*(ll - max))  (independent of the carried message)
    float m = llc[0];
#pragma unroll
    for (int q = 1; q < Q; ++q) m = fmaxf(m, llc[q]);
    m = group_max<WPC>(m, red, red_par, wig, lane, bar_id);
    float Lc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) Lc[q] = valid[q] ? __expf(scale * (llc[q] - m)) : 0.f;

    // a0 = (M^T alpha)_move, scaled for the Toeplitz factorisation P0 = diag(1/z) G
    float a0[Q], pr0[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) a0[q] = (M00 * al0[q] + M10 * al1[q]) * invz[q];
    band_apply<Q, WPC, WT>(a0, pr0, buf0 + par * bf, gl, tp, tapsS, c.tr.band_fwd, kind, W, K, bar_id);
    par ^= 1;

    float s2[2] = {0.f, 0.f};
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      al0[q] = pr0[q] * Lc[q];
      al1[q] = p1 * Lc[q];
      s2[0] += al0[q];
      s2[1] += al1[q];
    }
    group_sum<WPC, 2>(s2, red, red_par, wig, lane, bar_id);
    const float cn = s2[0] + s2[1];
    const float inv = 1.f / cn;
#pragma unroll
    for (int q = 0; q < Q; ++q) { al0[q] *= inv; al1[q] *= inv; }
    p1 = (M01 * s2[0] + M11 * s2[1]) * inv * invK;

    if (t >= cr.t_begin) {
      float* o = p.alpha + (size_t)t * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = al0[q];
          o[K + x] = al1[q];
        }
      }
      if (gl == 0) p.lmr[t] = logf(cn) + scale * m;
    } else if (t == cr.t_begin - 1 && p.halo_state) {
      float* o = p.halo_state + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = al0[q];
          o[K + x] = al1[q];
        }
      }
    }
    if (p.warm_out && t == cr.t_end - halo_next_of(c, cr.s + 1) - 1 && (cr.s + 1 < c.n_chain || !c.right_exact)) {
      float* o = p.warm_out + (size_t)(cr.s + 1) * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = al0[q];
          o[K + x] = al1[q];
        }
      }
    }
  }
}

// ============================================================================
// backward
// ============================================================================
template <int Q, int WPC, int WT>
__global__ void __launch_bounds__(256, 1) bwd_kernel(const BwdParams p) {
  using Ge = Geo<Q, WPC, WT>;
  extern __shared__ float smem[];
  const ScanCommon& c = p.c;
  if (cta_idle(c, Geo<Q, WPC, WT>::CPC)) return;
  const int K = c.tr.K, W = c.tr.W, kind = c.tr.kind;
  const int grp = threadIdx.x / Ge::G;
  const int gl = threadIdx.x % Ge::G;
  const int lane = threadIdx.x & 31;
  const int wig = gl >> 5;
  const int bar_id = 1 + grp;

  const int bf = Ge::buf_floats(W);
  float* buf0 = smem + (size_t)grp * (2 * bf + 2 * WPC * 4);
  float* red = buf0 + 2 * bf;
  float* tapsS = smem + (size_t)Ge::CPC * (2 * bf + 2 * WPC * 4);
  if (!Ge::REG) {
    if (kind == 0)
      for (int i = threadIdx.x; i <= W; i += blockDim.x) tapsS[i] = c.tr.taps[i];
  }
  for (int i = threadIdx.x; i < Ge::CPC * (2 * bf + 2 * WPC * 4); i += blockDim.x) smem[i] = 0.f;
  __syncthreads();

  ChainRange cr;
  if (!chain_range<Ge::CPC>(c, grp, cr)) return;

  float tp[2 * WT + 1];
  if constexpr (Ge::REG) {
#pragma unroll
    for (int j = 0; j <= 2 * WT; ++j) {
      const int d = j >= WT ? j - WT : WT - j;
      tp[j] = d <= W ? __ldg(c.tr.taps + d) : 0.f;
    }
  }
  float invz[Q];
  bool valid[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int x = own_x<Q, WPC, WT>(gl, q);
    valid[q] = x < K;
    invz[q] = (kind == 0 && valid[q]) ? __ldg(c.tr.inv_z + x) : 1.f;
  }
  const float M00 = c.tr.M00, M01 = c.tr.M01, M10 = c.tr.M10, M11 = c.tr.M11;
  const float invK = 1.f / (float)K;
  const float scale = c.scale;
  int red_par = 0;

  // ---- where the recursion starts
  int64_t t_hi;
  const float* init = bwd_start<true>(c, cr, p, t_hi, K);

  float be0[Q], be1[Q], Lb[Q], tw_acc[Q];
  float RL = 0.f;
#pragma unroll
  for (int q = 0; q < Q; ++q) { be0[q] = 0.f; be1[q] = 0.f; Lb[q] = 0.f; tw_acc[q] = 0.f; }

  // prefetch ll[t_hi] and alpha[t_hi] (alpha only where it is consumed)
  float lln[Q], an0[Q], an1[Q];
  {
    const float* row = c.ll + (size_t)t_hi * c.ldll;
    const bool need_a = t_hi <= cr.t_end && t_hi < c.T;
    const float* arow = p.alpha + (size_t)t_hi * 2 * K;
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      const int x = own_x<Q, WPC, WT>(gl, q);
      lln[q] = valid[q] ? __ldg(row + x) : -INFINITY;
      an0[q] = (need_a && valid[q]) ? __ldg(arow + x) : 0.f;
      an1[q] = (need_a && valid[q]) ? __ldg(arow + K + x) : 0.f;
    }
  }

  int par = 0;
  for (int64_t t = t_hi; t >= cr.t_begin; --t) {
    float llc[Q], ac0[Q], ac1[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) { llc[q] = lln[q]; ac0[q] = an0[q]; ac1[q] = an1[q]; }
    const bool use_alpha = t <= cr.t_end;   // core bins and the seam bin
    if (t - 1 >= cr.t_begin) {
      const float* row = c.ll + (size_t)(t - 1) * c.ldll;
      const bool need_a = (t - 1) <= cr.t_end;
      const float* arow = p.alpha + (size_t)(t - 1) * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x = own_x<Q, WPC, WT>(gl, q);
        lln[q] = valid[q] ? __ldg(row + x) : -INFINITY;
        an0[q] = (need_a && valid[q]) ? __ldg(arow + x) : 0.f;
        an1[q] = (need_a && valid[q]) ? __ldg(arow + K + x) : 0.f;
      }
    }
    float m = llc[0];
#pragma unroll
    for (int q = 1; q < Q; ++q) m = fmaxf(m, llc[q]);
    m = group_max<WPC>(m, red, red_par, wig, lane, bar_id);
    float Lc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) Lc[q] = valid[q] ? __expf(scale * (llc[q] - m)) : 0.f;

    // ---- unnormalised beta_t
    float b0[Q], b1[Q], r0[Q], r1[Q];
    if (t == t_hi) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x = own_x<Q, WPC, WT>(gl, q);
        b0[q] = valid[q] ? (init ? init[x] : 1.f) : 0.f;
        b1[q] = valid[q] ? (init ? init[K + x] : 1.f) : 0.f;
        r0[q] = 0.f; r1[q] = 0.f;
      }
    } else {
      float w0[Q];
#pragma unroll
      for (int q = 0; q < Q; ++q) { r0[q] = Lb[q] * be0[q]; r1[q] = Lb[q] * be1[q]; }
      band_apply<Q, WPC, WT>(r0, w0, buf0 + par * bf, gl, tp, tapsS, c.tr.band_bwd, kind, W, K, bar_id);
      par ^= 1;
      const float w1 = RL * invK;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const float w0q = w0[q] * invz[q];
        b0[q] = valid[q] ? (M00 * w0q + M01 * w1) : 0.f;
        b1[q] = valid[q] ? (M10 * w0q + M11 * w1) : 0.f;
      }
    }

    // ---- normaliser, fused with the jump-state sum for the next step
    float s3[3] = {0.f, 0.f, 0.f};
    if (use_alpha) {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        s3[0] = fmaf(ac0[q], b0[q], s3[0]);
        s3[1] = fmaf(ac1[q], b1[q], s3[1]);
        s3[2] = fmaf(Lc[q], b1[q], s3[2]);
      }
    } else {
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        s3[0] += b0[q];
        s3[1] += b1[q];
        s3[2] = fmaf(Lc[q], b1[q], s3[2]);
      }
    }
    group_sum<WPC, 3>(s3, red, red_par, wig, lane, bar_id);
    const float z = s3[0] + s3[1];
    const float inv = 1.f / z;
#pragma unroll
    for (int q = 0; q < Q; ++q) { be0[q] = b0[q] * inv; be1[q] = b1[q] * inv; Lb[q] = Lc[q]; }
    RL = s3[2] * inv;

    if (t < cr.t_end) {
      // core bin: posterior gamma_t = alpha_t * beta_t
      float* g = p.gamma ? p.gamma + (size_t)t * 2 * K : nullptr;
      float* gl_ = p.gamma_lat ? p.gamma_lat + (size_t)t * K : nullptr;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          const float g0 = ac0[q] * be0[q], g1 = ac1[q] * be1[q];
          if (g) { g[x] = g0; g[K + x] = g1; }
          if (gl_) gl_[x] = g0 + g1;
          if (p.gamma16) {
            const float gs = g0 + g1;
            const __half h = __float2half_rn(gs);
            p.gamma16[(size_t)t * p.ldg + x] = h;
            p.gamma16[((size_t)c.T + t) * p.ldg + x] = __float2half_rn(gs - __half2float(h));
          }
          tw_acc[q] += g0 + g1;
        }
      }
      if (p.dyn_marg && gl == 0) {
        p.dyn_marg[2 * t] = s3[0] * inv;
        p.dyn_marg[2 * t + 1] = s3[1] * inv;
      }
      if (p.r_out && t != t_hi) {
        float* ro = p.r_out + (size_t)(t + 1) * 2 * K;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          if (valid[q]) {
            const int x = own_x<Q, WPC, WT>(gl, q);
            ro[x] = r0[q] * inv;
            ro[K + x] = r1[q] * inv;
          }
        }
      }
    } else if (t == cr.t_end && p.beta_halo) {
      float* o = p.beta_halo + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = be0[q];
          o[K + x] = be1[q];
        }
      }
    }
    if (t == cr.t_begin && p.beta_end) {
      float* o = p.beta_end + (size_t)cr.s * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = be0[q];
          o[K + x] = be1[q];
        }
      }
    }
    if (p.warm_out && t == cr.t_begin + halo_next_of(c, cr.s - 1) - 1 && (cr.s >= 1 || !c.left_exact)) {
      float* o = p.warm_out + ((int64_t)cr.s - 1) * 2 * K;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        if (valid[q]) {
          const int x = own_x<Q, WPC, WT>(gl, q);
          o[x] = be0[q];
          o[K + x] = be1[q];
        }
      }
    }
  }
  if (p.tw_partial) {
    float* o = p.tw_partial + (size_t)cr.s * K;
#pragma unroll
    for (int q = 0; q < Q; ++q)
      if (valid[q]) o[own_x<Q, WPC, WT>(gl, q)] = tw_acc[q];
  }
}

// ============================================================================
// seam verification
// ============================================================================
// tol >= 0: seams with !(err <= tol) are counted into *counter (if given) and, with fix != 0, their estimate is
// overwritten by the truth: the snapshot a conditional restart (scan mode 2) of that chain starts from.
// One warp per seam (messages are 2K <= 8192 floats: two passes over L1-resident rows), 8 seams per CTA.
__global__ void __launch_bounds__(256) seam_check_kernel(int n, int len, float* est, int64_t ld_est, const float* truth,
                                                         int64_t ld_truth, float floor_val, float* err, float tol,
                                                         int fix, float* counter) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  float* a = est + (size_t)i * ld_est;
  const float* b = truth + (size_t)i * ld_truth;
  // messages are compared up to scale: normalise both to unit sum
  float sa = 0.f, sb = 0.f;
  for (int j = lane; j < len; j += 32) { sa += a[j]; sb += b[j]; }
  sa = warp_sum(sa); sb = warp_sum(sb);
  const float ia = 1.f / sa, ib = 1.f / sb;
  float e = 0.f;
  if (!(sa > 0.f) || !(sb > 0.f) || !(ia > 0.f) || !(ib > 0.f)) e = INFINITY;
  for (int j = lane; j < len; j += 32) {
    const float u = a[j] * ia, v = b[j] * ib;
    const float hi = fmaxf(u, v), lo = fminf(u, v);
    if (hi > floor_val) e = fmaxf(e, (hi - lo) / fmaxf(lo, 1e-37f));
    if (!(u == u) || !(v == v)) e = INFINITY;
  }
  e = warp_max(e);
  if (lane == 0) {
    err[i] = e;
    if (tol >= 0.f && !(e <= tol) && counter) atomicAdd(counter, 1.f);
  }
  if (tol >= 0.f && fix && !(e <= tol))
    for (int j = lane; j < len; j += 32) a[j] = b[j];
}

// ============================================================================
// host dispatch
// ============================================================================
template <int Q, int WPC, int WT>
static int launch_fwd(const FwdParams& p, int n_groups, cudaStream_t st) {
  using Ge = Geo<Q, WPC, WT>;
  const size_t smem = Ge::smem_bytes(p.c.tr.W);
  if (smem > 227 * 1024) return PMG_ERR_UNSUPPORTED_SHAPE;
  PMG_CUDA_CHECK(cudaFuncSetAttribute(fwd_kernel<Q, WPC, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fwd_kernel<Q, WPC, WT><<<cdiv(n_groups, Ge::CPC), 256, smem, st>>>(p);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
template <int Q, int WPC, int WT>
static int launch_bwd(const BwdParams& p, int n_groups, cudaStream_t st) {
  using Ge = Geo<Q, WPC, WT>;
  const size_t smem = Ge::smem_bytes(p.c.tr.W);
  if (smem > 227 * 1024) return PMG_ERR_UNSUPPORTED_SHAPE;
  PMG_CUDA_CHECK(cudaFuncSetAttribute(bwd_kernel<Q, WPC, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  bwd_kernel<Q, WPC, WT><<<cdiv(n_groups, Ge::CPC), 256, smem, st>>>(p);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

constexpr int kRegWT = 10;   // compile-time half width of the register-window Toeplitz path

}  // namespace pmg
#include "pmg_scan_bulk.cuh"
namespace pmg {

static bool wants_xi16(const FwdParams&) { return false; }
static bool wants_xi16(const BwdParams& p) { return p.xa_hi != nullptr; }
static bool bulk_ok(const FwdParams& p) {
  return (((uintptr_t)p.c.ll | (uintptr_t)p.alpha) & 15) == 0;
}
static bool bulk_ok(const BwdParams& p) {
  return (((uintptr_t)p.c.ll | (uintptr_t)p.alpha | (uintptr_t)p.gamma16) & 15) == 0;
}

template <bool FWD, int Q, int WT, int NW, int OB, typename P>
static int bulk_launch(const P& p, int n_groups, cudaStream_t st) {
  if constexpr (FWD) return launch_fwd_bulk<Q, WT, NW, OB>(p, n_groups, st);
  else return launch_bwd_bulk<Q, WT, NW, OB>(p, n_groups, st);
}
template <bool FWD, typename P>
static int dispatch(const P& p, int n_groups, cudaStream_t st) {
  const int K = p.c.tr.K;
  const bool reg = p.c.tr.kind == 0 && p.c.tr.W <= kRegWT;
  // whole-row bulk copies need 16-byte rows: K % 8 == 0 (fp16 posterior pieces), ld % 4 == 0
  // bulk kernels: 8 chains per CTA, double-buffered output staging (the best of 8/12/16 chains x 1/2 buffers
  // measured on B200)
  const bool w5 = p.c.tr.W <= 5;
  const bool bulk = reg && (K % 8 == 0) && (p.c.ldll % 4 == 0) && bulk_ok(p) && p.c.scale > 0.f;
  return by_tier(K, [&](auto Qc, auto WPCc) -> int {
    constexpr int Qv = Qc, WPCv = WPCc;
    if constexpr (WPCv == 1) {
      if (bulk) {
        const int rc = w5 ? bulk_launch<FWD, Qv, 5, 8, 2>(p, n_groups, st) : bulk_launch<FWD, Qv, 10, 8, 2>(p, n_groups, st);
        if (rc != PMG_ERR_UNSUPPORTED_SHAPE) return rc;
      }
    }
    if (wants_xi16(p)) return PMG_ERR_UNSUPPORTED_SHAPE;   // only the bulk kernel writes them
    if constexpr (FWD) return reg ? launch_fwd<Qv, WPCv, kRegWT>(p, n_groups, st) : launch_fwd<Qv, WPCv, 0>(p, n_groups, st);
    else return reg ? launch_bwd<Qv, WPCv, kRegWT>(p, n_groups, st) : launch_bwd<Qv, WPCv, 0>(p, n_groups, st);
  });
}

}  // namespace pmg

extern "C" int pmg_forward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                           const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                           float* alpha, float* lmr, float* halo_state, int mode,
                           const int* chain_ids, int n_ids, pmg_stream_t stream) {
  pmg::FwdParams p;
  int rc = pmg::fill_common(p.c, plan, tr, ll, ldll, mode, chain_ids, n_ids, true);
  if (rc) return rc;
  if (!alpha || !lmr) return PMG_ERR_BAD_ARG;
  p.carry_in = carry_in; p.warm_in = warm_in; p.warm_stride = warm_stride; p.warm_out = warm_out; p.alpha = alpha; p.lmr = lmr; p.halo_state = halo_state;
  const int n_groups = mode == 1 ? n_ids : plan->n_chain;
  return pmg::dispatch<true>(p, n_groups, (cudaStream_t)stream);
}

static int backward_impl(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                         const float* alpha, const float* beta_in, const float* warm_in, int64_t warm_stride,
                         float* warm_out, float* gamma, float* gamma_lat, void* gamma16, int64_t ldg, float* dyn_marg,
                         float* r_out, void* xa_hi, void* xa_lo, void* xr_hi, void* xr_lo, int64_t ld_x,
                         float* tw_partial, float* beta_halo, float* beta_end, int mode, const int* chain_ids, int n_ids,
                         pmg_stream_t stream) {
  pmg::BwdParams p;
  int rc = pmg::fill_common(p.c, plan, tr, ll, ldll, mode, chain_ids, n_ids, false);
  if (rc) return rc;
  if (xa_hi && !pmg_backward_xi16_supported(tr, plan->likelihood_scale)) return PMG_ERR_UNSUPPORTED_SHAPE;
  if (!alpha) return PMG_ERR_BAD_ARG;
  if (mode != 0 && !beta_end && !warm_in) return PMG_ERR_BAD_ARG;
  if (gamma16 && (ldg < tr->K || (ldg & 7))) return PMG_ERR_BAD_ARG;
  if (xa_hi) {
    if (!xa_lo || !xr_hi || !xr_lo || ld_x < 2 * tr->K || (ld_x & 7) || (tr->K & 7)) return PMG_ERR_BAD_ARG;
    if (((uintptr_t)xa_hi | (uintptr_t)xa_lo | (uintptr_t)xr_hi | (uintptr_t)xr_lo) & 15) return PMG_ERR_ALIGNMENT;
  }
  p.alpha = alpha; p.beta_in = beta_in; p.warm_in = warm_in; p.warm_stride = warm_stride; p.warm_out = warm_out;
  p.gamma = gamma; p.gamma_lat = gamma_lat; p.dyn_marg = dyn_marg;
  p.gamma16 = (__half*)gamma16; p.ldg = ldg;
  p.r_out = r_out; p.tw_partial = tw_partial; p.beta_halo = beta_halo; p.beta_end = beta_end;
  p.xa_hi = (uint16_t*)xa_hi; p.xa_lo = (uint16_t*)xa_lo; p.xr_hi = (uint16_t*)xr_hi; p.xr_lo = (uint16_t*)xr_lo;
  p.ld_x = ld_x;
  const int n_groups = mode == 1 ? n_ids : plan->n_chain;
  return pmg::dispatch<false>(p, n_groups, (cudaStream_t)stream);
}

extern "C" int pmg_backward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                            const float* alpha, const float* beta_in, const float* warm_in, int64_t warm_stride,
                            float* warm_out, float* gamma, float* gamma_lat,
                            void* gamma16, int64_t ldg, float* dyn_marg, float* r_out, float* tw_partial, float* beta_halo,
                            float* beta_end, int mode, const int* chain_ids, int n_ids,
                            pmg_stream_t stream) {
  return backward_impl(plan, tr, ll, ldll, alpha, beta_in, warm_in, warm_stride, warm_out, gamma, gamma_lat, gamma16, ldg,
                       dyn_marg, r_out, nullptr, nullptr, nullptr, nullptr, 0, tw_partial, beta_halo, beta_end, mode,
                       chain_ids, n_ids, stream);
}

extern "C" int pmg_backward_xi16_supported(const pmg_transition* tr, float likelihood_scale) {
  // the conditions under which dispatch<false> takes the bulk kernel (pointer alignment is checked at the call)
  return tr && tr->kind == 0 && tr->W <= pmg::kRegWT && tr->K % 8 == 0 && tr->K <= 32 * 16 && likelihood_scale > 0.f;
}

extern "C" int pmg_backward_xi16(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                                 const float* alpha, const float* beta_in, const float* warm_in, int64_t warm_stride,
                                 float* warm_out, float* gamma, float* gamma_lat, void* gamma16, int64_t ldg,
                                 float* dyn_marg, void* xa_hi, void* xa_lo, void* xr_hi, void* xr_lo, int64_t ld_x,
                                 float* tw_partial, float* beta_halo, float* beta_end, int mode, const int* chain_ids,
                                 int n_ids, pmg_stream_t stream) {
  if (!xa_hi) return PMG_ERR_BAD_ARG;
  return backward_impl(plan, tr, ll, ldll, alpha, beta_in, warm_in, warm_stride, warm_out, gamma, gamma_lat, gamma16, ldg,
                       dyn_marg, nullptr, xa_hi, xa_lo, xr_hi, xr_lo, ld_x, tw_partial, beta_halo, beta_end, mode,
                       chain_ids, n_ids, stream);
}

extern "C" int pmg_seam_check(int n, int len, const float* est, int64_t ld_est, const float* truth,
                              int64_t ld_truth, float floor_val, float* err, pmg_stream_t stream) {
  if (n <= 0) return PMG_OK;
  if (!est || !truth || !err || len <= 0) return PMG_ERR_BAD_ARG;
  pmg::seam_check_kernel<<<(n + 7) / 8, 256, 0, (cudaStream_t)stream>>>(n, len, const_cast<float*>(est), ld_est, truth,
                                                                        ld_truth, floor_val, err, -1.f, 0, nullptr);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_seam_check_fix(int n, int len, float* est, int64_t ld_est, const float* truth, int64_t ld_truth,
                                  float floor_val, float tol, int fix, float* err, float* counter,
                                  pmg_stream_t stream) {
  if (n <= 0) return PMG_OK;
  if (!est || !truth || !err || len <= 0 || !(tol >= 0.f)) return PMG_ERR_BAD_ARG;
  pmg::seam_check_kernel<<<(n + 7) / 8, 256, 0, (cudaStream_t)stream>>>(n, len, est, ld_est, truth, ld_truth, floor_val,
                                                                        err, tol, fix, counter);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

#include "pmg_scan_pk.cuh"
