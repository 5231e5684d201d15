// Adam M-step of the per-neuron Poisson GLM on the GP basis, one persistent
// cooperative kernel for the whole optimisation loop.
//
// Replaces reference poor_man_gplvm/fit_tuning_helper.py:124-196 (make_adam_runner.run:
// optax.adam + lax.while_loop with the global relative-loss stop rule) on the
// objective :63-81 (poisson_m_step_objective) with the softplus link :19-25.
//   loss(W) = -sum_{k,n} [ xlogy(yw, pf+1e-20) - pf*tw_k ] - sum logN(W; 0, sigma),  pf = softplus(Phi W)
//   dL/dW   = -Phi^T [ (yw/(pf+1e-20) - tw) * sigmoid(Phi W) ] + W / sigma^2      (column separable)
// The gradient is separable per neuron, so each CTA owns tiles of NT neurons; the
// only grid-wide quantity is the scalar loss (and the reported gradient norm),
// exchanged once per step through per-CTA partial slots and a counter barrier.
#include <cooperative_groups.h>

#include "pmg_common.cuh"
#include <cstdlib>

namespace pmg {

constexpr int MS_NT = 4;        // neurons per tile
constexpr int MS_THREADS = 256;

// the gradient phase splits the K rows of Phi into this many parts, one thread per (part, basis function)
__host__ __device__ constexpr int mstep_parts(int threads, int B) { return B >= threads ? 1 : threads / B; }

struct MstepParams {
  int K, B, N;
  const float* Phi;
  const float* yw;       // [K, ldyw]
  const float* tw;       // element k at tw[k * tws]
  int64_t ldyw, tws;
  float prior_std, lr, b1, b2, eps;
  int maxiter;
  float tol;
  int min_iters;
  float* W;
  float* mu;
  float* nu;
  int* count;
  float* loss_hist;
  float* err_hist;
  int* n_iter_out;
  float* final_out;
  float* tuning_out;
  double* partials;      // [maxiter][grid][2]
  unsigned* barrier;
  int phi_in_smem;
  int Bs;                // smem row stride of Phi (odd)
};

__device__ __forceinline__ void grid_barrier(unsigned* ctr, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(ctr, 1u);
    while (*(volatile unsigned*)ctr < target) { }
    __threadfence();
  }
  __syncthreads();
}

__global__ void __launch_bounds__(MS_THREADS, 1) mstep_adam_kernel(const MstepParams p) {
  extern __shared__ float smem[];
  const int K = p.K, B = p.B, N = p.N, Bs = p.Bs;
  const int tid = threadIdx.x;
  float* phiS = smem;                                   // [K][Bs] when phi_in_smem
  float* wS = phiS + (p.phi_in_smem ? (((size_t)K * Bs + 3) & ~(size_t)3) : 0);   // [B][NT], 16B aligned
  float* eS = wS + (size_t)B * MS_NT;                   // [K][NT]
  const int parts = mstep_parts(MS_THREADS, B);
  float* gS = eS + (size_t)K * MS_NT;                   // [parts][B][NT]
  __shared__ double redD[2][MS_THREADS / 32];
  __shared__ float bcast[4];

  if (p.phi_in_smem) {
    for (int i = tid; i < K * B; i += MS_THREADS) phiS[(size_t)(i / B) * Bs + (i % B)] = p.Phi[i];
  }
  __syncthreads();
  const float* phi = p.phi_in_smem ? phiS : p.Phi;
  const int ldphi = p.phi_in_smem ? Bs : B;

  const int ntiles = (N + MS_NT - 1) / MS_NT;
  const float inv_s2 = 1.f / (p.prior_std * p.prior_std);
  const float log_norm = logf(6.283185307179586f * p.prior_std * p.prior_std);
  const int count0 = *p.count;

  // evaluates loss/gradient at the current W for every tile of this CTA; applies one Adam
  // update when `update` (optax: mu,nu EMA, bias correction with the incremented count).
  auto eval = [&](bool update, int step_count, double& loss_cta, double& err_cta, bool write_tuning) {
    loss_cta = 0.0; err_cta = 0.0;
    const float bc1 = 1.f - powf(p.b1, (float)step_count);
    const float bc2 = 1.f - powf(p.b2, (float)step_count);
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
      const int n0 = tile * MS_NT;
      for (int i = tid; i < B * MS_NT; i += MS_THREADS) {
        const int b = i / MS_NT, nt = i % MS_NT;
        wS[i] = (n0 + nt < N) ? p.W[(size_t)b * N + n0 + nt] : 0.f;
      }
      __syncthreads();
      // phase 1: rows of Phi -> z, pf, residual e, likelihood part of the loss
      float loss_t = 0.f;
      for (int k = tid; k < K; k += MS_THREADS) {
        float z[MS_NT];
#pragma unroll
        for (int nt = 0; nt < MS_NT; ++nt) z[nt] = 0.f;
        const float* prow = phi + (size_t)k * ldphi;
        for (int b = 0; b < B; ++b) {
          const float ph = prow[b];
          const float4 w4 = *reinterpret_cast<const float4*>(wS + b * MS_NT);
          z[0] = fmaf(ph, w4.x, z[0]); z[1] = fmaf(ph, w4.y, z[1]);
          z[2] = fmaf(ph, w4.z, z[2]); z[3] = fmaf(ph, w4.w, z[3]);
        }
        const float twk = p.tw[(size_t)k * p.tws];
#pragma unroll
        for (int nt = 0; nt < MS_NT; ++nt) {
          float e = 0.f;
          if (n0 + nt < N) {
            const float pf = softplus_f(z[nt]);
            if (write_tuning) {
              p.tuning_out[(size_t)k * N + n0 + nt] = pf;
            } else {
              const float ywv = p.yw[(size_t)k * p.ldyw + n0 + nt];
              const float pfe = pf + kLamFloor;
              e = (ywv / pfe - twk) * sigmoid_f(z[nt]);
              const float fit = (ywv == 0.f) ? 0.f : ywv * logf(pfe);
              loss_t -= fit - pf * twk;
            }
          }
          eS[k * MS_NT + nt] = e;
        }
      }
      if (write_tuning) { __syncthreads(); continue; }
      __syncthreads();
      // phase 2: g[b,nt] = sum_k Phi[k,b] e[k,nt], k split into `parts`
      if (B >= MS_THREADS) {
        for (int b = tid; b < B; b += MS_THREADS) {
          float g[MS_NT] = {0.f, 0.f, 0.f, 0.f};
          for (int k = 0; k < K; ++k) {
            const float ph = phi[(size_t)k * ldphi + b];
            const float4 e4 = *reinterpret_cast<const float4*>(eS + k * MS_NT);
            g[0] = fmaf(ph, e4.x, g[0]); g[1] = fmaf(ph, e4.y, g[1]);
            g[2] = fmaf(ph, e4.z, g[2]); g[3] = fmaf(ph, e4.w, g[3]);
          }
#pragma unroll
          for (int nt = 0; nt < MS_NT; ++nt) gS[b * MS_NT + nt] = g[nt];
        }
      } else if (tid < parts * B) {
        const int part = tid / B, b = tid % B;
        const int kb = (int)(((int64_t)K * part) / parts), ke = (int)(((int64_t)K * (part + 1)) / parts);
        float g[MS_NT] = {0.f, 0.f, 0.f, 0.f};
        for (int k = kb; k < ke; ++k) {
          const float ph = phi[(size_t)k * ldphi + b];
          const float4 e4 = *reinterpret_cast<const float4*>(eS + k * MS_NT);
          g[0] = fmaf(ph, e4.x, g[0]); g[1] = fmaf(ph, e4.y, g[1]);
          g[2] = fmaf(ph, e4.z, g[2]); g[3] = fmaf(ph, e4.w, g[3]);
        }
#pragma unroll
        for (int nt = 0; nt < MS_NT; ++nt) gS[((size_t)part * B + b) * MS_NT + nt] = g[nt];
      }
      __syncthreads();
      // phase 3: gradient, prior, Adam
      float err_t = 0.f;
      for (int i = tid; i < B * MS_NT; i += MS_THREADS) {
        const int b = i / MS_NT, nt = i % MS_NT;
        if (n0 + nt >= N) continue;
        float gsum = 0.f;
        for (int pz = 0; pz < parts; ++pz) gsum += gS[((size_t)pz * B + b) * MS_NT + nt];
        const float w = wS[i];
        const float g = -gsum + w * inv_s2;
        err_t = fmaf(g, g, err_t);
        loss_t += 0.5f * (log_norm + w * w * inv_s2);
        if (update) {
          const size_t gi = (size_t)b * N + n0 + nt;
          const float m = p.b1 * p.mu[gi] + (1.f - p.b1) * g;
          const float v = p.b2 * p.nu[gi] + (1.f - p.b2) * g * g;
          p.mu[gi] = m; p.nu[gi] = v;
          p.W[gi] = w - p.lr * ((m / bc1) / (sqrtf(v / bc2) + p.eps));
        }
      }
      loss_cta += (double)loss_t;     // per-thread partials, reduced below
      err_cta += (double)err_t;
      __syncthreads();
    }
  };

  auto cta_publish = [&](int slot, double loss_thr, double err_thr) {
    double a = warp_sum_d(loss_thr), b = warp_sum_d(err_thr);
    if ((tid & 31) == 0) { redD[0][tid >> 5] = a; redD[1][tid >> 5] = b; }
    __syncthreads();
    if (tid == 0) {
      double s0 = 0.0, s1 = 0.0;
      for (int w = 0; w < MS_THREADS / 32; ++w) { s0 += redD[0][w]; s1 += redD[1][w]; }
      p.partials[((size_t)slot * gridDim.x + blockIdx.x) * 2 + 0] = s0;
      p.partials[((size_t)slot * gridDim.x + blockIdx.x) * 2 + 1] = s1;
    }
  };
  auto gather = [&](int slot, float& loss, float& err) {
    if (tid < 32) {
      // one warp, fixed order (lane-strided partial sums, then a butterfly): every CTA computes the
      // same bits, so all CTAs take the same stop decision
      double s0 = 0.0, s1 = 0.0;
      const double* src = p.partials + (size_t)slot * gridDim.x * 2;
      for (unsigned c = tid; c < gridDim.x; c += 32) {
        s0 += __ldcg(src + 2 * c);
        s1 += __ldcg(src + 2 * c + 1);
      }
      s0 = warp_sum_d(s0);
      s1 = warp_sum_d(s1);
      if (tid == 0) {
        bcast[0] = (float)s0;
        bcast[1] = sqrtf((float)s1);
      }
    }
    __syncthreads();
    loss = bcast[0]; err = bcast[1];
    __syncthreads();
  };

  double lc, ec;
  unsigned bar = 0;
  eval(false, count0 + 1, lc, ec, false);
  cta_publish(0, lc, ec);
  grid_barrier(p.barrier, ++bar * gridDim.x);
  float loss, err;
  gather(0, loss, err);
  float loss_prev = loss;
  if (blockIdx.x == 0 && tid == 0) { p.loss_hist[0] = loss; p.err_hist[0] = err; }
  int i = 0;
  while (true) {
    const float rel = fabsf(loss - loss_prev) / fmaxf(fabsf(loss), 1e-8f);
    if (!(i < p.maxiter - 1 && (i < p.min_iters || rel > p.tol))) break;
    eval(true, count0 + i + 1, lc, ec, false);
    cta_publish(i + 1, lc, ec);
    grid_barrier(p.barrier, ++bar * gridDim.x);
    float nl, ne;
    gather(i + 1, nl, ne);
    ++i;
    if (blockIdx.x == 0 && tid == 0) { p.loss_hist[i] = nl; p.err_hist[i] = ne; }
    loss_prev = loss; loss = nl; err = ne;
  }
  if (blockIdx.x == 0 && tid == 0) {
    *p.n_iter_out = i + 1;
    *p.count = count0 + i;
    p.final_out[0] = loss;
    p.final_out[1] = err;
  }
  if (p.tuning_out) eval(false, 1, lc, ec, true);
}

// ---------------------------------------------------------------------------------------------------
// Same optimisation with the grid-wide reduction taken off the critical path.
//
// The gradient is separable per neuron; only the STOP decision needs the global loss.  Every CTA therefore
// keeps stepping on its own tile while the loss of step j is reduced: it publishes its partial of every step
// (per-step slots + per-step arrival counters) and evaluates the reference's stop rule for step i - LAG, by
// which time all partials of that step have long arrived.  The last LAG+1 optimiser states (W, mu, nu) of the
// tile live in shared memory; when the rule says "stop before update j", the state after j updates is
// restored.  The per-element arithmetic, the fixed reduction order of the partials and the stop rule are those of
// mstep_adam_kernel, but with 512 instead of 256 threads the gradient's K sum is split into 512/B instead of 256/B
// parts and each thread sums the loss over other rows: the two kernels agree to fp32 rounding, not bit for bit.  A
// rule that rounding cannot decide (tol < 0, a stop at min_iters) stops both at the same step.  One tile per CTA
// (N <= 4 * #resident CTAs), state of a tile in shared memory.
// ---------------------------------------------------------------------------------------------------
constexpr int MS_LAG = 4;        // a step's stop rule is evaluated at least this many steps later
constexpr int MS_BATCH = 4;      // ... and MS_BATCH steps at a time (one warp per step)

template <int LT>
__global__ void __launch_bounds__(LT, 1) mstep_adam_lag_kernel(const MstepParams p, unsigned* arrived) {
  extern __shared__ float smem[];
  const int K = p.K, B = p.B, N = p.N, Bs = p.Bs;
  const int tid = threadIdx.x;
  constexpr int R = MS_LAG + MS_BATCH + 1;
  const int BT = B * MS_NT;
  float* phiS = smem;                                   // [K][Bs] when phi_in_smem
  float* eS = phiS + (p.phi_in_smem ? (((size_t)K * Bs + 3) & ~(size_t)3) : 0);   // [K][NT], 16B aligned
  const int parts = mstep_parts(LT, B);
  float* gS = eS + (size_t)K * MS_NT;                   // [parts][B][NT]
  float* ywS = gS + (size_t)parts * BT;                 // [K][NT]
  float* twS = ywS + (size_t)K * MS_NT;                 // [K]
  float* Wr = twS + ((K + 3) & ~3);                     // [R][B][NT] ring of optimiser states
  float* Mr = Wr + (size_t)R * BT;
  float* Vr = Mr + (size_t)R * BT;
  __shared__ double redD[2][2][LT / 32];            // [step parity][loss, err][warp]
  __shared__ float bL[MS_BATCH], bE[MS_BATCH];

  const int n0 = blockIdx.x * MS_NT;
  if (p.phi_in_smem) {
    for (int i = tid; i < K * B; i += LT) phiS[(size_t)(i / B) * Bs + (i % B)] = p.Phi[i];
  }
  for (int i = tid; i < BT; i += LT) {
    const int b = i / MS_NT, nt = i % MS_NT;
    const bool ok = n0 + nt < N;
    const size_t gi = (size_t)b * N + n0 + nt;
    Wr[i] = ok ? p.W[gi] : 0.f;
    Mr[i] = ok ? p.mu[gi] : 0.f;
    Vr[i] = ok ? p.nu[gi] : 0.f;
  }
  for (int i = tid; i < K * MS_NT; i += LT) {
    const int k = i / MS_NT, nt = i % MS_NT;
    ywS[i] = (n0 + nt < N) ? p.yw[(size_t)k * p.ldyw + n0 + nt] : 0.f;
  }
  for (int k = tid; k < K; k += LT) twS[k] = p.tw[(size_t)k * p.tws];
  __syncthreads();
  const float* phi = p.phi_in_smem ? phiS : p.Phi;
  const int ldphi = p.phi_in_smem ? Bs : B;
  const float inv_s2 = 1.f / (p.prior_std * p.prior_std);
  const float log_norm = logf(6.283185307179586f * p.prior_std * p.prior_std);
  const int count0 = *p.count;

  // loss / gradient at ring state `cur`; with `update` the Adam step goes to ring state `nxt`
  auto eval = [&](int cur, int nxt, bool update, int step_count, double& loss_cta, double& err_cta,
                  bool write_tuning) {
    const float bc1 = 1.f - powf(p.b1, (float)step_count);
    const float bc2 = 1.f - powf(p.b2, (float)step_count);
    const float* wS = Wr + (size_t)cur * BT;
    float loss_t = 0.f;
    for (int k = tid; k < K; k += LT) {
      float z[MS_NT];
#pragma unroll
      for (int nt = 0; nt < MS_NT; ++nt) z[nt] = 0.f;
      const float* prow = phi + (size_t)k * ldphi;
      for (int b = 0; b < B; ++b) {
        const float ph = prow[b];
        const float4 w4 = *reinterpret_cast<const float4*>(wS + b * MS_NT);
        z[0] = fmaf(ph, w4.x, z[0]); z[1] = fmaf(ph, w4.y, z[1]);
        z[2] = fmaf(ph, w4.z, z[2]); z[3] = fmaf(ph, w4.w, z[3]);
      }
      const float twk = twS[k];
#pragma unroll
      for (int nt = 0; nt < MS_NT; ++nt) {
        float e = 0.f;
        if (n0 + nt < N) {
          const float pf = softplus_f(z[nt]);
          if (write_tuning) {
            p.tuning_out[(size_t)k * N + n0 + nt] = pf;
          } else {
            const float ywv = ywS[k * MS_NT + nt];
            const float pfe = pf + kLamFloor;
            e = (ywv / pfe - twk) * sigmoid_f(z[nt]);
            const float fit = (ywv == 0.f) ? 0.f : ywv * logf(pfe);
            loss_t -= fit - pf * twk;
          }
        }
        eS[k * MS_NT + nt] = e;
      }
    }
    if (write_tuning) return;
    __syncthreads();
    if (B >= LT) {
      for (int b = tid; b < B; b += LT) {
        float g[MS_NT] = {0.f, 0.f, 0.f, 0.f};
        for (int k = 0; k < K; ++k) {
          const float ph = phi[(size_t)k * ldphi + b];
          const float4 e4 = *reinterpret_cast<const float4*>(eS + k * MS_NT);
          g[0] = fmaf(ph, e4.x, g[0]); g[1] = fmaf(ph, e4.y, g[1]);
          g[2] = fmaf(ph, e4.z, g[2]); g[3] = fmaf(ph, e4.w, g[3]);
        }
#pragma unroll
        for (int nt = 0; nt < MS_NT; ++nt) gS[b * MS_NT + nt] = g[nt];
      }
    } else if (tid < parts * B) {
      const int part = tid / B, b = tid % B;
      const int kb = (int)(((int64_t)K * part) / parts), ke = (int)(((int64_t)K * (part + 1)) / parts);
      float g[MS_NT] = {0.f, 0.f, 0.f, 0.f};
      for (int k = kb; k < ke; ++k) {
        const float ph = phi[(size_t)k * ldphi + b];
        const float4 e4 = *reinterpret_cast<const float4*>(eS + k * MS_NT);
        g[0] = fmaf(ph, e4.x, g[0]); g[1] = fmaf(ph, e4.y, g[1]);
        g[2] = fmaf(ph, e4.z, g[2]); g[3] = fmaf(ph, e4.w, g[3]);
      }
#pragma unroll
      for (int nt = 0; nt < MS_NT; ++nt) gS[((size_t)part * B + b) * MS_NT + nt] = g[nt];
    }
    __syncthreads();
    float err_t = 0.f;
    for (int i = tid; i < BT; i += LT) {
      const int nt = i % MS_NT;
      if (n0 + nt >= N) continue;
      const int b = i / MS_NT;
      float gsum = 0.f;
      for (int pz = 0; pz < parts; ++pz) gsum += gS[((size_t)pz * B + b) * MS_NT + nt];
      const float w = wS[i];
      const float g = -gsum + w * inv_s2;
      err_t = fmaf(g, g, err_t);
      loss_t += 0.5f * (log_norm + w * w * inv_s2);
      if (update) {
        const float m = p.b1 * Mr[(size_t)cur * BT + i] + (1.f - p.b1) * g;
        const float v = p.b2 * Vr[(size_t)cur * BT + i] + (1.f - p.b2) * g * g;
        Mr[(size_t)nxt * BT + i] = m; Vr[(size_t)nxt * BT + i] = v;
        Wr[(size_t)nxt * BT + i] = w - p.lr * ((m / bc1) / (sqrtf(v / bc2) + p.eps));
      }
    }
    loss_cta = (double)loss_t;      // per-thread partials, reduced by publish()
    err_cta = (double)err_t;
  };

  // per-CTA partial of a step -> its slot, then the step's arrival counter.  The last thread publishes (its warp
  // has no rows of Phi in phase 1 when K <= LT - 32), nobody waits for its fence: the staging is double-buffered
  // by step parity and the ring writes of this step are ordered by the barrier below.
  auto publish = [&](int slot, double loss_thr, double err_thr) {
    const int par = slot & 1;
    double a = warp_sum_d(loss_thr), b = warp_sum_d(err_thr);
    if ((tid & 31) == 0) { redD[par][0][tid >> 5] = a; redD[par][1][tid >> 5] = b; }
    __syncthreads();
    if (tid == LT - 1) {
      double s0 = 0.0, s1 = 0.0;
      for (int w = 0; w < LT / 32; ++w) { s0 += redD[par][0][w]; s1 += redD[par][1][w]; }
      p.partials[((size_t)slot * gridDim.x + blockIdx.x) * 2 + 0] = s0;
      p.partials[((size_t)slot * gridDim.x + blockIdx.x) * 2 + 1] = s1;
      __threadfence();
      atomicAdd(arrived + slot, 1u);
    }
  };
  // global loss / gradient norm of steps first .. first+n-1, one warp per step (waits for every CTA's partial;
  // fixed summation order: the same bits in every CTA, hence the same decisions)
  auto resolve = [&](int first, int n) {
    const int w = tid >> 5, ln = tid & 31;
    if (w < n) {
      const int slot = first + w;
      if (ln == 0) {
        while (*(volatile unsigned*)(arrived + slot) < gridDim.x) { }
        __threadfence();
      }
      __syncwarp();
      double s0 = 0.0, s1 = 0.0;
      const double* src = p.partials + (size_t)slot * gridDim.x * 2;
      for (unsigned c = ln; c < gridDim.x; c += 32) {
        s0 += __ldcg(src + 2 * c);
        s1 += __ldcg(src + 2 * c + 1);
      }
      s0 = warp_sum_d(s0);
      s1 = warp_sum_d(s1);
      if (ln == 0) { bL[w] = (float)s0; bE[w] = sqrtf((float)s1); }
    }
    __syncthreads();
  };

  double lc, ec;
  eval(0, 0, false, count0 + 1, lc, ec, false);
  publish(0, lc, ec);
  int done = 0;                     // updates performed by this CTA (slots 0 .. done are published)
  int decided = 0;                  // stop rule evaluated for steps 0 .. decided-1 (all said "continue")
  int stop_at = -1;
  float l_prev = 0.f, l_fin = 0.f, e_fin = 0.f;
  while (stop_at < 0) {
    // rules are evaluated MS_BATCH steps at a time once the newest of them is MS_LAG steps old (and for every
    // remaining step once no further update is possible)
    const bool drain = done >= p.maxiter - 1;
    while (stop_at < 0 && (decided + MS_BATCH - 1 <= done - MS_LAG || drain)) {
      int n = done - decided + 1;
      if (n > MS_BATCH) n = MS_BATCH;
      resolve(decided, n);
      for (int j = 0; j < n && stop_at < 0; ++j) {
        const float l = bL[j], e = bE[j];
        if (blockIdx.x == 0 && tid == 0) { p.loss_hist[decided] = l; p.err_hist[decided] = e; }
        // reference loop: at its first test loss_prev == loss
        const float rel = decided == 0 ? 0.f : fabsf(l - l_prev) / fmaxf(fabsf(l), 1e-8f);
        const bool cont = decided < p.maxiter - 1 && (decided < p.min_iters || rel > p.tol);
        l_prev = l;
        if (!cont) { stop_at = decided; l_fin = l; e_fin = e; }
        else ++decided;
      }
      __syncthreads();              // bL / bE are rewritten by the next batch
    }
    if (stop_at >= 0) break;
    eval(done % R, (done + 1) % R, true, count0 + done + 1, lc, ec, false);
    publish(done + 1, lc, ec);
    ++done;
  }
  // state after stop_at updates
  const int fin = stop_at % R;
  for (int i = tid; i < BT; i += LT) {
    const int b = i / MS_NT, nt = i % MS_NT;
    if (n0 + nt >= N) continue;
    const size_t gi = (size_t)b * N + n0 + nt;
    p.W[gi] = Wr[(size_t)fin * BT + i];
    p.mu[gi] = Mr[(size_t)fin * BT + i];
    p.nu[gi] = Vr[(size_t)fin * BT + i];
  }
  if (blockIdx.x == 0 && tid == 0) {
    *p.n_iter_out = stop_at + 1;
    *p.count = count0 + stop_at;
    p.final_out[0] = l_fin;
    p.final_out[1] = e_fin;
  }
  if (p.tuning_out) eval(fin, fin, false, 1, lc, ec, true);
}

template <int LT>
static size_t mstep_lag_smem(int K, int B, bool phi_in_smem, int Bs) {
  const int parts = mstep_parts(LT, B);
  size_t f = (size_t)K * MS_NT + (size_t)parts * B * MS_NT + (size_t)K * MS_NT + (size_t)((K + 3) & ~3) +
             (size_t)3 * (MS_LAG + MS_BATCH + 1) * B * MS_NT;
  if (phi_in_smem) f += ((size_t)K * Bs + 3) & ~(size_t)3;
  return f * sizeof(float);
}

// tuning = softplus(Phi W): small standalone kernel (used outside the M-step)
__global__ void tuning_softplus_kernel(int K, int B, int N, const float* __restrict__ Phi,
                                       const float* __restrict__ W, float* __restrict__ tuning) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)K * N) return;
  const int k = (int)(i / N), n = (int)(i % N);
  float z = 0.f;
  for (int b = 0; b < B; ++b) z = fmaf(Phi[(size_t)k * B + b], W[(size_t)b * N + n], z);
  tuning[i] = softplus_f(z);
}

static size_t mstep_smem(int K, int B, bool phi_in_smem, int Bs) {
  const int parts = mstep_parts(MS_THREADS, B);
  size_t f = (size_t)B * MS_NT + (size_t)K * MS_NT + (size_t)parts * B * MS_NT;
  if (phi_in_smem) f += ((size_t)K * Bs + 3) & ~(size_t)3;
  return f * sizeof(float);
}

constexpr int MS_LAG_THREADS = 512;   // threads per CTA of the lagged kernel (one round over K <= 512 rows of Phi)

struct MstepPlan {
  int lagged;          // 1: mstep_adam_lag_kernel, 0: mstep_adam_kernel
  int phi_in_smem, Bs, grid, parts;
  size_t smem;
};

// Kernel, placement of Phi and grid of an M-step launch on the current device.  pmg_mstep_adam_ld launches what this
// returns and pmg_mstep_plan reports it.  Sets the chosen kernel's dynamic shared-memory limit, which the occupancy
// query and the launch need.
static int mstep_plan(int K, int B, int N, MstepPlan& pl) {
  pl.Bs = B | 1;
  pl.phi_in_smem = mstep_smem(K, B, true, pl.Bs) <= 200 * 1024;
  pl.smem = mstep_smem(K, B, pl.phi_in_smem, pl.Bs);
  if (pl.smem > 227 * 1024) return PMG_ERR_UNSUPPORTED_SHAPE;
  const int ntiles = (N + MS_NT - 1) / MS_NT;
  int dev = 0, sms = 0;
  PMG_CUDA_CHECK(cudaGetDevice(&dev));
  PMG_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  {
    // lagged-decision kernel: one tile per CTA, all CTAs resident, tile state + operands in shared memory
    const char* lag_s = std::getenv("PMG_MSTEP_LAG");      // 0 = the barrier-per-step kernel (cross-check)
    const int lag_env = lag_s ? std::atoi(lag_s) : 1;
    constexpr int LT = MS_LAG_THREADS;
    const bool phi_l = mstep_lag_smem<LT>(K, B, true, pl.Bs) <= 200 * 1024;
    const size_t smem_l = mstep_lag_smem<LT>(K, B, phi_l, pl.Bs);
    if (lag_env && smem_l <= 200 * 1024) {
      // attribute + occupancy query once per shared-memory size (host time of a launch that runs every EM iteration)
      static size_t cached_smem = 0;
      static int cached_per = 0, cached_dev = -1;
      if (cached_smem != smem_l || cached_dev != dev) {
        cached_dev = dev;
        PMG_CUDA_CHECK(cudaFuncSetAttribute(mstep_adam_lag_kernel<LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_l));
        PMG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cached_per, mstep_adam_lag_kernel<LT>, LT, smem_l));
        cached_smem = smem_l;
      }
      if (cached_per >= 1 && ntiles <= sms * cached_per && ntiles <= 1024) {
        pl.lagged = 1; pl.phi_in_smem = phi_l; pl.smem = smem_l; pl.grid = ntiles; pl.parts = mstep_parts(LT, B);
        return PMG_OK;
      }
    }
  }
  PMG_CUDA_CHECK(cudaFuncSetAttribute(mstep_adam_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  int per_sm = 0;
  PMG_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mstep_adam_kernel, MS_THREADS, pl.smem));
  if (per_sm < 1) return PMG_ERR_UNSUPPORTED_SHAPE;
  pl.lagged = 0;
  pl.grid = sms * per_sm;
  if (pl.grid > ntiles) pl.grid = ntiles;
  if (pl.grid > 1024) pl.grid = 1024;
  pl.parts = mstep_parts(MS_THREADS, B);
  return PMG_OK;
}

}  // namespace pmg

extern "C" int64_t pmg_mstep_workspace_bytes(int K, int B, int N, int maxiter) {
  (void)K; (void)B; (void)N;
  // barrier word (256-byte header) + partials for up to 1024 CTAs + per-step arrival counters
  return 256 + (int64_t)(maxiter + 1) * 1024 * 2 * (int64_t)sizeof(double) + (int64_t)(maxiter + 1) * 4 + 256;
}

extern "C" int pmg_mstep_plan(int K, int B, int N, int maxiter, int* kernel, int* phi_in_smem, int* grid, int* parts) {
  if (K <= 0 || B <= 0 || N <= 0 || maxiter < 1) return PMG_ERR_BAD_ARG;
  pmg::MstepPlan pl;
  const int rc = pmg::mstep_plan(K, B, N, pl);
  if (rc != PMG_OK) return rc;
  if (kernel) *kernel = pl.lagged;
  if (phi_in_smem) *phi_in_smem = pl.phi_in_smem;
  if (grid) *grid = pl.grid;
  if (parts) *parts = pl.parts;
  return PMG_OK;
}

extern "C" int pmg_mstep_adam(int K, int B, int N, const float* Phi, const float* yw, const float* tw,
                              float prior_std, float lr, float b1, float b2, float eps, int maxiter, float tol,
                              int min_iters, float* W, float* mu, float* nu, int* count, float* loss_hist,
                              float* err_hist, int* n_iter_out, float* final_out, float* tuning_out,
                              void* workspace, int64_t workspace_bytes, pmg_stream_t stream) {
  return pmg_mstep_adam_ld(K, B, N, Phi, yw, N, tw, 1, prior_std, lr, b1, b2, eps, maxiter, tol, min_iters, W, mu, nu,
                           count, loss_hist, err_hist, n_iter_out, final_out, tuning_out, workspace, workspace_bytes,
                           stream);
}

extern "C" int pmg_mstep_adam_ld(int K, int B, int N, const float* Phi, const float* yw, int64_t ldyw,
                                 const float* tw, int64_t tw_stride,
                                 float prior_std, float lr, float b1, float b2, float eps, int maxiter, float tol,
                                 int min_iters, float* W, float* mu, float* nu, int* count, float* loss_hist,
                                 float* err_hist, int* n_iter_out, float* final_out, float* tuning_out,
                                 void* workspace, int64_t workspace_bytes, pmg_stream_t stream) {
  using namespace pmg;
  if (K <= 0 || B <= 0 || N <= 0 || maxiter < 1 || ldyw < N || tw_stride < 1) return PMG_ERR_BAD_ARG;
  if (!Phi || !yw || !tw || !W || !mu || !nu || !count || !loss_hist || !err_hist || !n_iter_out || !final_out)
    return PMG_ERR_BAD_ARG;
  if (!workspace || workspace_bytes < pmg_mstep_workspace_bytes(K, B, N, maxiter)) return PMG_ERR_WORKSPACE;
  MstepPlan pl;
  const int rc = mstep_plan(K, B, N, pl);
  if (rc != PMG_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;

  MstepParams p;
  p.K = K; p.B = B; p.N = N; p.Phi = Phi; p.yw = yw; p.tw = tw; p.ldyw = ldyw; p.tws = tw_stride;
  p.prior_std = prior_std; p.lr = lr; p.b1 = b1; p.b2 = b2; p.eps = eps;
  p.maxiter = maxiter; p.tol = tol; p.min_iters = min_iters;
  p.W = W; p.mu = mu; p.nu = nu; p.count = count; p.loss_hist = loss_hist; p.err_hist = err_hist;
  p.n_iter_out = n_iter_out; p.final_out = final_out; p.tuning_out = tuning_out;
  p.barrier = (unsigned*)workspace;
  p.partials = (double*)((char*)workspace + 256);
  p.Bs = pl.Bs;
  p.phi_in_smem = pl.phi_in_smem;

  PMG_CUDA_CHECK(cudaMemsetAsync(workspace, 0, 256, st));
  PMG_CUDA_CHECK(cudaMemsetAsync(loss_hist, 0, sizeof(float) * maxiter, st));
  PMG_CUDA_CHECK(cudaMemsetAsync(err_hist, 0, sizeof(float) * maxiter, st));
  if (pl.lagged) {
    unsigned* arrived = (unsigned*)((char*)workspace + 256 + (size_t)(maxiter + 1) * 1024 * 2 * sizeof(double));
    PMG_CUDA_CHECK(cudaMemsetAsync(arrived, 0, (size_t)(maxiter + 1) * sizeof(unsigned), st));
    void* args_l[] = {(void*)&p, (void*)&arrived};
    PMG_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)mstep_adam_lag_kernel<MS_LAG_THREADS>, dim3(pl.grid),
                                               dim3(MS_LAG_THREADS), args_l, pl.smem, st));
  } else {
    void* args[] = {(void*)&p};
    PMG_CUDA_CHECK(cudaLaunchCooperativeKernel((const void*)mstep_adam_kernel, dim3(pl.grid), dim3(MS_THREADS), args,
                                               pl.smem, st));
  }
  return PMG_OK;
}

extern "C" int pmg_tuning_softplus(int K, int B, int N, const float* Phi, const float* W, float* tuning,
                                   pmg_stream_t stream) {
  if (K <= 0 || B <= 0 || N <= 0 || !Phi || !W || !tuning) return PMG_ERR_BAD_ARG;
  pmg::tuning_softplus_kernel<<<pmg::cdiv((int64_t)K * N, 256), 256, 0, (cudaStream_t)stream>>>(K, B, N, Phi, W, tuning);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
