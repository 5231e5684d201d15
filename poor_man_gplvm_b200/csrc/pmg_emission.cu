// Poisson emission log-likelihood in GEMM form and the naive-Bayes normalisation.
//
// Replaces reference poor_man_gplvm/decoder.py:30-48 (get_loglikelihood_ma_poisson),
// :60-85 (its vmap over time) and :88-102 (get_naive_bayes_ma):
//   ll[t,k] = sum_n y[t,n] * (ma_n log lam[k,n]) - sum_n ma_n lam[k,n] - sum_n ma_n lgamma(y[t,n]+1)
// with lam = tuning*dt + 1e-20 and ll = -1e20 on masked latent bins.
#include "pmg_common.cuh"

namespace pmg {

// one CTA per latent bin k
__global__ void emission_prepare_kernel(int K, int N, const float* __restrict__ tuning,
                                        const float* __restrict__ ma_neuron, float dt,
                                        float* __restrict__ loglam, float* __restrict__ lam_sum) {
  const int k = blockIdx.x;
  double acc = 0.0;
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    const float m = ma_neuron ? ma_neuron[n] : 1.f;
    const float lam = tuning[(size_t)k * N + n] * dt + kLamFloor;
    loglam[(size_t)k * N + n] = m * logf(lam);
    acc += (double)(m * lam);
  }
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

// one warp per time bin
// ma_neuron: NULL, a vector (ldm = 0) or a [T,N] matrix (ldm = row stride, decoder.py:291-294);
// ysum (optional): masked row sums of the counts (needed by the per-bin dt path, decoder.py:73-85)
__global__ void lgamma_rowsum_kernel(int64_t T, int N, const float* __restrict__ y, int64_t ldy,
                                     const float* __restrict__ ma_neuron, int64_t ldm, float* __restrict__ out,
                                     float* __restrict__ ysum) {
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const int lane = threadIdx.x & 31;
  const float* row = y + (size_t)t * ldy;
  const float* mrow = ma_neuron ? ma_neuron + (size_t)t * ldm : nullptr;
  float acc = 0.f, ys = 0.f;
  for (int n = lane; n < N; n += 32) {
    const float v = row[n];
    // lgamma(1) = lgamma(2) = 0: skip the (dominant) 0/1 counts
    const float lg = (v == 0.f || v == 1.f) ? 0.f : lgammaf(v + 1.f);
    const float m = mrow ? mrow[n] : 1.f;
    acc += m * lg;
    ys += m * v;
  }
  acc = warp_sum(acc);
  ys = warp_sum(ys);
  if (lane == 0) {
    out[t] = acc;
    if (ysum) ysum[t] = ys;
  }
}

// Augmented right-hand operands for the option surface that the plain GEMM form does not cover:
//  mode 1, [T,N] neuron mask m (decoder.py:291-294): with A = [m*y | m] the product with
//          B[k,:] = [log lam_k | -lam_k] gives sum_n m (y log lam - lam); lam_sum = 0.
//  mode 2, per-bin dt (decoder.py:73-85): log(tun*dt + 1e-20) = log dt + log(tun + 1e-20/dt); with
//          A = [y | dt_t] and B[k,:] = [ma log(tun_k + 1e-20) | -sum_n ma tun_kn] the product gives the
//          dt-dependent part; lam_sum = 1e-20 * sum_n ma.  Exact up to the position of the 1e-20 floor
//          (relative effect <= 1e-20 |1 - 1/dt| / tun).
// out: [rows_out, ldo] fp32, rows >= K and columns past the operand are zero.  One CTA per row.
__global__ void emission_prepare_aug_kernel(int K, int N, const float* __restrict__ tuning,
                                            const float* __restrict__ ma_neuron, float dt, int mode,
                                            float* __restrict__ out, int64_t ldo, float* __restrict__ lam_sum) {
  const int k = blockIdx.x;
  float* o = out + (size_t)k * ldo;
  if (k >= K) {
    for (int n = threadIdx.x; n < (int)ldo; n += blockDim.x) o[n] = 0.f;
    return;
  }
  const int ncol = mode == 1 ? 2 * N : N + 1;
  double acc = 0.0, msum = 0.0;
  for (int n = threadIdx.x; n < N; n += blockDim.x) {
    const float tun = tuning[(size_t)k * N + n];
    if (mode == 1) {
      const float lam = tun * dt + kLamFloor;
      o[n] = logf(lam);
      o[N + n] = -lam;
    } else {
      const float m = ma_neuron ? ma_neuron[n] : 1.f;
      o[n] = m * logf(tun + kLamFloor);
      acc += (double)(m * tun);
      msum += (double)m;
    }
  }
  for (int n = ncol + threadIdx.x; n < (int)ldo; n += blockDim.x) o[n] = 0.f;
  acc = warp_sum_d(acc);
  msum = warp_sum_d(msum);
  __shared__ double sm[2][32];
  if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = acc; sm[1][threadIdx.x >> 5] = msum; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0, ms = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { s += sm[0][w]; ms += sm[1][w]; }
    if (mode == 1) {
      lam_sum[k] = 0.f;
    } else {
      o[N] = -(float)s;
      lam_sum[k] = (float)(ms * (double)kLamFloor);
    }
  }
}

// ---- CUDA-core fp32 tile GEMM with the emission epilogue: used when the counts are not exactly
// representable in fp16 (non-integer "counts", decoder.py:37-38) and as the cross-check of the tcgen05 kernel ----
constexpr int EM_BM = 128, EM_BN = 64, EM_BK = 16;

__global__ void __launch_bounds__(256) emission_simt_kernel(int64_t T, int N, int K,
                                                            const float* __restrict__ y, int64_t ldy,
                                                            const float* __restrict__ loglam,
                                                            const float* __restrict__ lam_sum,
                                                            const float* __restrict__ lgam,
                                                            const float* __restrict__ ma_latent,
                                                            float* __restrict__ ll, int64_t ldll) {
  __shared__ float As[EM_BK][EM_BM + 4];
  __shared__ float Bs[EM_BK][EM_BN + 4];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int64_t t0 = (int64_t)blockIdx.x * EM_BM;
  const int k0 = blockIdx.y * EM_BN;
  float acc[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  for (int n0 = 0; n0 < N; n0 += EM_BK) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 4, cc = idx & 15;
      const int64_t t = t0 + r;
      const int n = n0 + cc;
      As[cc][r] = (t < T && n < N) ? y[(size_t)t * ldy + n] : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 4, cc = idx & 15;
      const int k = k0 + r;
      const int n = n0 + cc;
      Bs[cc][r] = (k < K && n < N) ? loglam[(size_t)k * N + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < EM_BK; ++kk) {
      float a[8], b[4];
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = As[kk][ty * 8 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t t = t0 + ty * 8 + i;
    if (t >= T) continue;
    const float lg = lgam[t];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= K) continue;
      float v = acc[i][j] - lam_sum[k] - lg;
      if (ma_latent && ma_latent[k] == 0.f) v = kVeryNegLL;
      ll[(size_t)t * ldll + k] = v;
    }
  }
}

// ---- Gaussian observation model (reference decoder.py:50-57, SURVEY F2): ll[t,k] = sum_n m (-(y - mu_kn)^2 / (2 s^2)
// - log(2 pi s^2) / 2).  Same tiling as the fp32 emission GEMM with the squared difference as the inner operation
// (the expanded GEMM form y mu - mu^2/2 cancels catastrophically in fp32 for real-valued observations).
// ma: NULL, a vector [N] (ld_mask = 0) or a [T, ld_mask] mask. ----
__global__ void __launch_bounds__(256) emission_gaussian_kernel(int64_t T, int N, int K,
                                                                const float* __restrict__ y, int64_t ldy,
                                                                const float* __restrict__ mu,
                                                                const float* __restrict__ ma, int64_t ld_mask,
                                                                float inv_2var, float half_log_2pivar,
                                                                const float* __restrict__ ma_latent,
                                                                float* __restrict__ ll, int64_t ldll) {
  __shared__ float As[EM_BK][EM_BM + 4];
  __shared__ float Ws[EM_BK][EM_BM + 4];
  __shared__ float Bs[EM_BK][EM_BN + 4];
  const int tid = threadIdx.x;
  const int ty = tid >> 4, tx = tid & 15;
  const int64_t t0 = (int64_t)blockIdx.x * EM_BM;
  const int k0 = blockIdx.y * EM_BN;
  float acc[8][4], wsum[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    wsum[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  }
  for (int n0 = 0; n0 < N; n0 += EM_BK) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 4, cc = idx & 15;
      const int64_t t = t0 + r;
      const int n = n0 + cc;
      const bool ok = t < T && n < N;
      As[cc][r] = ok ? y[(size_t)t * ldy + n] : 0.f;
      float w = 0.f;
      if (ok) w = !ma ? 1.f : (ld_mask ? ma[(size_t)t * ld_mask + n] : ma[n]);
      Ws[cc][r] = w;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = tid + i * 256;
      const int r = idx >> 4, cc = idx & 15;
      const int k = k0 + r;
      const int n = n0 + cc;
      Bs[cc][r] = (k < K && n < N) ? mu[(size_t)k * N + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < EM_BK; ++kk) {
      float a[8], w[8], b[4];
#pragma unroll
      for (int i = 0; i < 8; ++i) { a[i] = As[kk][ty * 8 + i]; w[i] = Ws[kk][ty * 8 + i]; wsum[i] += w[i]; }
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float d = a[i] - b[j];
          acc[i][j] = fmaf(w[i] * d, d, acc[i][j]);
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t t = t0 + ty * 8 + i;
    if (t >= T) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= K) continue;
      float v = -inv_2var * acc[i][j] - half_log_2pivar * wsum[i];
      if (ma_latent && ma_latent[k] == 0.f) v = kVeryNegLL;
      ll[(size_t)t * ldll + k] = v;
    }
  }
}

// logsumexp_k row[k] by one warp (every lane gets the result); shared by both naive-Bayes kernels so that their
// lml_t agree bit for bit
__device__ __forceinline__ float nb_row_logsumexp(const float* __restrict__ row, int K, int lane) {
  float m = -INFINITY;
  for (int k = lane; k < K; k += 32) m = fmaxf(m, row[k]);
  m = warp_max(m);
  if (!(fabsf(m) <= 3.0e38f)) m = 0.f;   // jax logsumexp: non-finite max -> 0
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s += expf(row[k] - m);
  s = warp_sum(s);
  return logf(s) + m;
}

// one warp per time bin: lml = logsumexp_k ll, log_post = ll - lml
__global__ void nb_normalize_kernel(int64_t T, int K, const float* __restrict__ ll, int64_t ldll,
                                    float* __restrict__ log_post, int64_t ldp, float* __restrict__ lml_t,
                                    float* __restrict__ post) {
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const int lane = threadIdx.x & 31;
  const float* row = ll + (size_t)t * ldll;
  const float lml = nb_row_logsumexp(row, K, lane);
  float* orow = log_post + (size_t)t * ldp;
  float* prow = post ? post + (size_t)t * ldp : nullptr;
  for (int k = lane; k < K; k += 32) {
    const float lp = row[k] - lml;
    orow[k] = lp;
    if (prow) prow[k] = expf(lp);            // posterior_latent = exp(log_posterior_latent), core.py:517
  }
  if (lane == 0) lml_t[t] = lml;
}

// the log marginal alone (shuffle tests read nothing else): a read-only pass over ll
__global__ void nb_lml_kernel(int64_t T, int K, const float* __restrict__ ll, int64_t ldll,
                              float* __restrict__ lml_t) {
  const int64_t t = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= T) return;
  const int lane = threadIdx.x & 31;
  const float lml = nb_row_logsumexp(ll + (size_t)t * ldll, K, lane);
  if (lane == 0) lml_t[t] = lml;
}

}  // namespace pmg

extern "C" int pmg_emission_prepare(int K, int N, const float* tuning, const float* ma_neuron, float dt,
                                    float* loglam, float* lam_sum, pmg_stream_t stream) {
  if (K <= 0 || N <= 0 || !tuning || !loglam || !lam_sum) return PMG_ERR_BAD_ARG;
  pmg::emission_prepare_kernel<<<K, 128, 0, (cudaStream_t)stream>>>(K, N, tuning, ma_neuron, dt, loglam, lam_sum);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_gaussian(int64_t T, int N, int K, const float* y, int64_t ldy, const float* mu,
                                     const float* ma_neuron, int64_t ld_mask, float noise_std, const float* ma_latent,
                                     float* ll, int64_t ldll, pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || K <= 0 || !y || !mu || !ll || ldy < N || ldll < K || !(noise_std > 0.f)) return PMG_ERR_BAD_ARG;
  if (ld_mask != 0 && ld_mask < N) return PMG_ERR_BAD_ARG;
  const float var = noise_std * noise_std;
  dim3 grid((unsigned)pmg::cdiv(T, pmg::EM_BM), (unsigned)pmg::cdiv(K, pmg::EM_BN));
  pmg::emission_gaussian_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(
      T, N, K, y, ldy, mu, ma_neuron, ld_mask, 0.5f / var, 0.5f * logf(6.283185307179586f * var), ma_latent, ll, ldll);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_lgamma_rowsum(int64_t T, int N, const float* y, int64_t ldy,
                                          const float* ma_neuron, float* lgam, pmg_stream_t stream) {
  return pmg_emission_row_terms(T, N, y, ldy, ma_neuron, 0, lgam, nullptr, stream);
}

extern "C" int pmg_emission_row_terms(int64_t T, int N, const float* y, int64_t ldy, const float* ma_neuron,
                                      int64_t ld_mask, float* lgam, float* ysum, pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || !y || !lgam || ldy < N) return PMG_ERR_BAD_ARG;
  if (ma_neuron && ld_mask != 0 && ld_mask < N) return PMG_ERR_BAD_ARG;
  pmg::lgamma_rowsum_kernel<<<pmg::cdiv(T, 8), 256, 0, (cudaStream_t)stream>>>(T, N, y, ldy, ma_neuron, ld_mask,
                                                                              lgam, ysum);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_prepare_aug(int K, int N, const float* tuning, const float* ma_neuron, float dt,
                                        int mode, int rows_out, float* out, int64_t ldo, float* lam_sum,
                                        pmg_stream_t stream) {
  if (K <= 0 || N <= 0 || !tuning || !out || !lam_sum || rows_out < K) return PMG_ERR_BAD_ARG;
  if (mode != 1 && mode != 2) return PMG_ERR_BAD_ARG;
  if (ldo < (mode == 1 ? 2 * (int64_t)N : (int64_t)N + 1)) return PMG_ERR_BAD_ARG;
  pmg::emission_prepare_aug_kernel<<<rows_out, 128, 0, (cudaStream_t)stream>>>(K, N, tuning, ma_neuron, dt, mode,
                                                                              out, ldo, lam_sum);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_emission_poisson(int64_t T, int N, int K, const float* y, int64_t ldy, const float* loglam,
                                    const float* lam_sum, const float* lgam, const float* ma_latent, float* ll,
                                    int64_t ldll, pmg_stream_t stream) {
  if (T <= 0 || N <= 0 || K <= 0 || !y || !loglam || !lam_sum || !lgam || !ll) return PMG_ERR_BAD_ARG;
  if (ldy < N || ldll < K) return PMG_ERR_BAD_ARG;
  dim3 grid(pmg::cdiv(T, pmg::EM_BM), pmg::cdiv(K, pmg::EM_BN));
  pmg::emission_simt_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(T, N, K, y, ldy, loglam, lam_sum, lgam,
                                                                   ma_latent, ll, ldll);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_naive_bayes_normalize(int64_t T, int K, const float* ll, int64_t ldll, float* log_post,
                                         int64_t ldp, float* lml_t, pmg_stream_t stream) {
  if (T <= 0 || K <= 0 || !ll || !log_post || !lml_t || ldll < K || ldp < K) return PMG_ERR_BAD_ARG;
  pmg::nb_normalize_kernel<<<pmg::cdiv(T, 8), 256, 0, (cudaStream_t)stream>>>(T, K, ll, ldll, log_post, ldp, lml_t,
                                                                            nullptr);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_naive_bayes_lml(int64_t T, int K, const float* ll, int64_t ldll, float* lml_t,
                                   pmg_stream_t stream) {
  if (T <= 0 || K <= 0 || !ll || !lml_t || ldll < K) return PMG_ERR_BAD_ARG;
  pmg::nb_lml_kernel<<<pmg::cdiv(T, 8), 256, 0, (cudaStream_t)stream>>>(T, K, ll, ldll, lml_t);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_naive_bayes_posterior(int64_t T, int K, const float* ll, int64_t ldll, float* log_post,
                                         float* post, int64_t ldp, float* lml_t, pmg_stream_t stream) {
  if (T <= 0 || K <= 0 || !ll || !log_post || !post || !lml_t || ldll < K || ldp < K) return PMG_ERR_BAD_ARG;
  pmg::nb_normalize_kernel<<<pmg::cdiv(T, 8), 256, 0, (cudaStream_t)stream>>>(T, K, ll, ldll, log_post, ldp, lml_t,
                                                                            post);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
