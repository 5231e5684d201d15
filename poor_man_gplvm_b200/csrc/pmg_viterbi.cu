// Viterbi decoding of the joint (dynamics, latent) HMM, parallel in time over the chains of pmg_forward.
//
// Beyond the reference (which decodes marginals only).  The forward pass is the max-product analogue of
// fwd_kernel (pmg_scan.cu): same chain plan, warm-ups, warm-start messages and repair modes, with the band SUM of
// the move operator replaced by a band MAX that also records its argmax.  Messages are normalised by their sum
// every step, as in the filter, so the seam messages have the filter's scale and pmg_seam_check_fix applies as is.
// Backpointers hold the flat predecessor state d*K + x as int16; exact ties go to the smallest flat index.
//
// The backtrack is time-parallel too: pmg_viterbi_chain_maps follows, for every chain and every end state, the
// backpointers through the chain's core (maps[c, s] = state at the chain's first bin); pmg_viterbi_backtrack then
// resolves the chain end states from last to first (n_chain dependent lookups) and lets every chain fill its core.
//
// Time-sharded runs keep backpointers for the rank's own bins only.  pmg_viterbi_block_link summarises a rank's block
// as a map from its end state to the left neighbour's end state; the ranks all-gather those maps (with the last
// messages), and pmg_viterbi_backtrack_sharded resolves this rank's end state from the last rank's argmax before it
// backtracks its own chains as pmg_viterbi_backtrack does.
#include <climits>

#include "pmg_common.cuh"

namespace pmg {
namespace vit {

struct Params {
  int64_t T, core_begin, core_end, chunk_len;
  int n_chain, halo, halo_next, left_exact, right_exact;
  const int* halo_arr;
  const int* halo_next_arr;
  const float* sel_err;
  float sel_tol;
  float scale;
  int K, kind, W;
  const float* taps;
  const float* inv_z;
  const float* band_fwd;
  float M00, M01, M10, M11;
  const float* ll;
  int64_t ldll;
  const float* carry_in;
  const float* warm_in;
  int64_t warm_stride;
  float* warm_out;
  int16_t* bp;
  int64_t ldbp;
  float* lmr;
  float* halo_state;
  float* end_msg;
  int mode;
  const int* chain_ids;
  int n_ids;
};

// (value, flat index) order of the max-product: larger value first, then the smaller index
__device__ __forceinline__ bool better(float v, int i, float bv, int bi) { return v > bv || (v == bv && i < bi); }

__device__ __forceinline__ void warp_argmax(float& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, o);
    const int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (better(ov, oi, v, i)) { v = ov; i = oi; }
  }
}

template <int WPC>
__device__ __forceinline__ void group_argmax(float& v, int& i, float* red, int& red_par, int wig, int lane,
                                             int bar_id) {
  warp_argmax(v, i);
  if (WPC > 1) {
    float* r = red + red_par * (WPC * 4);
    if (lane == 0) { r[wig * 4] = v; r[wig * 4 + 1] = __int_as_float(i); }
    named_bar_sync(bar_id, 32 * WPC);
    float bv = r[0];
    int bi = __float_as_int(r[1]);
#pragma unroll
    for (int w = 1; w < WPC; ++w) {
      const float ov = r[w * 4];
      const int oi = __float_as_int(r[w * 4 + 1]);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    v = bv; i = bi;
    red_par ^= 1;
  }
}

template <int WPC>
__device__ __forceinline__ void group_sum2(float (&v)[2], float* red, int& red_par, int wig, int lane, int bar_id) {
  v[0] = warp_sum(v[0]);
  v[1] = warp_sum(v[1]);
  if (WPC > 1) {
    float* r = red + red_par * (WPC * 4);
    if (lane == 0) { r[wig * 4] = v[0]; r[wig * 4 + 1] = v[1]; }
    named_bar_sync(bar_id, 32 * WPC);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int w = 0; w < WPC; ++w) { s0 += r[w * 4]; s1 += r[w * 4 + 1]; }
    v[0] = s0; v[1] = s1;
    red_par ^= 1;
  }
}

template <int WPC>
__device__ __forceinline__ float group_max(float v, float* red, int& red_par, int wig, int lane, int bar_id) {
  v = warp_max(v);
  if (WPC > 1) {
    float* r = red + red_par * (WPC * 4);
    if (lane == 0) r[wig * 4] = v;
    named_bar_sync(bar_id, 32 * WPC);
    float s = r[0];
#pragma unroll
    for (int w = 1; w < WPC; ++w) s = fmaxf(s, r[w * 4]);
    v = s;
    red_par ^= 1;
  }
  return v;
}

template <int WPC>
__device__ __forceinline__ void group_sync(int bar_id) {
  if (WPC > 1) named_bar_sync(bar_id, 32 * WPC);
  else __syncwarp();
}

__device__ __forceinline__ int16_t as_state(int i, int K2) { return (int16_t)((unsigned)i < (unsigned)K2 ? i : 0); }

template <int Q, int WPC>
struct Geo {
  static constexpr int G = 32 * WPC;     // threads per chain; thread gl owns bins gl + G*q
  static constexpr int CPC = 8 / WPC;    // chains per 256-thread CTA
  static constexpr int KP = G * Q;
  // per chain: 2 value + 2 index exchange buffers of KP + 2W entries (padded by W on each side), reduction scratch
  __host__ __device__ static int buf(int W) { return KP + 2 * W; }
  __host__ __device__ static int per_chain(int W) { return 4 * buf(W) + 2 * WPC * 4; }
  __host__ __device__ static size_t smem_bytes(int W) { return sizeof(float) * ((size_t)CPC * per_chain(W) + W + 1); }
};

template <int Q, int WPC>
__global__ void __launch_bounds__(256, 1) viterbi_fwd_kernel(const Params p) {
  using Ge = Geo<Q, WPC>;
  extern __shared__ float smem[];
  if (p.mode == 2) {   // no chain of this CTA selected: return before touching shared memory
    int any = 0;
    for (int j = threadIdx.x; j < Ge::CPC; j += blockDim.x) {
      const int s = blockIdx.x * Ge::CPC + j;
      if (s < p.n_chain && !(p.sel_err[s] <= p.sel_tol)) any = 1;
    }
    if (__syncthreads_or(any) == 0) return;
  }
  const int K = p.K, W = p.W, kind = p.kind, K2 = 2 * K;
  const int grp = threadIdx.x / Ge::G;
  const int gl = threadIdx.x % Ge::G;
  const int lane = threadIdx.x & 31;
  const int wig = gl >> 5;
  const int bar_id = 1 + grp;
  const int bf = Ge::buf(W), pc = Ge::per_chain(W);
  float* vbuf = smem + (size_t)grp * pc;        // [2][bf] values (padding -1: never a maximum)
  int* ibuf = (int*)(vbuf + 2 * bf);            // [2][bf] flat predecessor indices
  float* red = vbuf + 4 * bf;
  float* tapsS = smem + (size_t)Ge::CPC * pc;
  if (kind == 0)
    for (int i = threadIdx.x; i <= W; i += blockDim.x) tapsS[i] = p.taps[i];
  for (int i = threadIdx.x; i < Ge::CPC * pc; i += blockDim.x) {
    const int o = i % pc;
    if (o < 2 * bf) smem[i] = -1.f;
    else if (o < 4 * bf) ((int*)smem)[i] = INT_MAX;
    else smem[i] = 0.f;
  }
  __syncthreads();

  // ---- chain of this group (mode 1: listed chains; mode 2: selected on the device)
  int s;
  {
    const int idx = blockIdx.x * Ge::CPC + grp;
    if (p.mode == 1) {
      if (idx >= p.n_ids) return;
      s = p.chain_ids[idx];
    } else {
      s = idx;
    }
    if (s < 0 || s >= p.n_chain) return;
    if (p.mode == 2 && p.sel_err[s] <= p.sel_tol) return;
  }
  const int64_t t_begin = p.core_begin + (int64_t)s * p.chunk_len;
  int64_t t_end = t_begin + p.chunk_len;
  if (t_end > p.core_end) t_end = p.core_end;
  if (t_begin >= t_end) return;

  float invz[Q];
  bool valid[Q];
#pragma unroll
  for (int q = 0; q < Q; ++q) {
    const int x = gl + Ge::G * q;
    valid[q] = x < K;
    invz[q] = (kind == 0 && valid[q]) ? __ldg(p.inv_z + x) : 1.f;
  }
  const float M00 = p.M00, M01 = p.M01, M10 = p.M10, M11 = p.M11;
  const float invK = 1.f / (float)K;
  const float scale = p.scale;
  int red_par = 0;

  // ---- initial message: the carry in front of bin 0, or a warm start (pmg_forward's conventions)
  int64_t t0;
  const float* src = nullptr;
  if (p.mode != 0) {
    t0 = t_begin;
    src = t0 > 0 ? p.warm_in + (size_t)s * p.warm_stride : p.carry_in;
  } else {
    const int h = p.halo_arr ? p.halo_arr[s] : p.halo;
    t0 = t_begin - h;
    if (t0 <= 0 && p.left_exact) {
      t0 = 0;
      src = p.carry_in;
    } else {
      if (t0 < 0) t0 = 0;
      if (p.warm_in) src = p.warm_in + (size_t)s * p.warm_stride;
    }
  }
  float de0[Q], de1[Q];   // the normalised message delta-hat (move, jump)
  float p1 = 0.f;         // jump-state prior of a sum-product step (bin 0)
  {
    bool ok = false;
    if (src) {
      float s2[2] = {0.f, 0.f};
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x = gl + Ge::G * q;
        de0[q] = valid[q] ? src[x] : 0.f;
        de1[q] = valid[q] ? src[K + x] : 0.f;
        s2[0] += de0[q];
        s2[1] += de1[q];
      }
      group_sum2<WPC>(s2, red, red_par, wig, lane, bar_id);
      const float tot = s2[0] + s2[1];
      if (tot > 0.f && tot < 3.0e38f) {
        const float inv = 1.f / tot;
#pragma unroll
        for (int q = 0; q < Q; ++q) { de0[q] *= inv; de1[q] *= inv; }
        p1 = (M01 * s2[0] + M11 * s2[1]) * inv * invK;
        ok = true;
      }
    }
    if (!ok) {   // no or unusable initial message: uniform
      const float u = 0.5f * invK;
#pragma unroll
      for (int q = 0; q < Q; ++q) { de0[q] = valid[q] ? u : 0.f; de1[q] = de0[q]; }
      p1 = (M01 * 0.5f + M11 * 0.5f) * invK;
    }
  }

  float lln[Q];
  {
    const float* row = p.ll + (size_t)t0 * p.ldll;
#pragma unroll
    for (int q = 0; q < Q; ++q) lln[q] = valid[q] ? __ldg(row + gl + Ge::G * q) : -INFINITY;
  }

  int par = 0;
  for (int64_t t = t0; t < t_end; ++t) {
    float llc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) llc[q] = lln[q];
    if (t + 1 < t_end) {
      const float* row = p.ll + (size_t)(t + 1) * p.ldll;
#pragma unroll
      for (int q = 0; q < Q; ++q) lln[q] = valid[q] ? __ldg(row + gl + Ge::G * q) : -INFINITY;
    }
    float m = llc[0];
#pragma unroll
    for (int q = 1; q < Q; ++q) m = fmaxf(m, llc[q]);
    m = group_max<WPC>(m, red, red_par, wig, lane, bar_id);
    float Lc[Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) Lc[q] = valid[q] ? __expf(scale * (llc[q] - m)) : 0.f;

    float* vb = vbuf + par * bf;
    int* ib = ibuf + par * bf;
    par ^= 1;
    float pr0[Q], pr1;
    int ix0[Q], ix1 = 0;
    if (t == 0) {
      // bin 0: the start is marginalised -- the filter's prior from the carry (sum over the band)
#pragma unroll
      for (int q = 0; q < Q; ++q)
        vb[W + gl + Ge::G * q] = valid[q] ? (M00 * de0[q] + M10 * de1[q]) * invz[q] : -1.f;
      group_sync<WPC>(bar_id);
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x1 = gl + Ge::G * q;
        float acc = 0.f;
        if (valid[q]) {
          for (int j = 0; j <= 2 * W; ++j) {
            const int x = x1 - W + j;
            if ((unsigned)x >= (unsigned)K) continue;
            const float w = kind == 0 ? tapsS[j >= W ? j - W : W - j] : __ldg(p.band_fwd + (size_t)j * K + x1);
            acc = fmaf(w, vb[x1 + j], acc);
          }
        }
        pr0[q] = acc;
        ix0[q] = 0;
      }
      pr1 = p1;
    } else {
      // a_{d'}[x] = max_d delta[d,x] M[d,d'] (ties: d = 0); the jump target's prior is one scalar
      float b1v = -1.f;
      int b1i = INT_MAX;
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x = gl + Ge::G * q;
        const float v00 = de0[q] * M00, v10 = de1[q] * M10;
        const float v01 = de0[q] * M01, v11 = de1[q] * M11;
        const bool j0 = v10 > v00, j1 = v11 > v01;
        const float a0 = j0 ? v10 : v00, a1 = j1 ? v11 : v01;
        vb[W + x] = valid[q] ? a0 * invz[q] : -1.f;
        ib[W + x] = valid[q] ? (j0 ? K + x : x) : INT_MAX;
        if (valid[q] && better(a1, j1 ? K + x : x, b1v, b1i)) { b1v = a1; b1i = j1 ? K + x : x; }
      }
      group_argmax<WPC>(b1v, b1i, red, red_par, wig, lane, bar_id);
      pr1 = b1v * invK;
      ix1 = b1i;
      group_sync<WPC>(bar_id);
      // band max of the move target: prior_0[x'] = max_{x in band} a_0[x] P0[x,x']
#pragma unroll
      for (int q = 0; q < Q; ++q) {
        const int x1 = gl + Ge::G * q;
        float bv = -INFINITY;
        int bi = valid[q] ? ib[x1 + W] : INT_MAX;
        if (valid[q]) {
          if (kind == 0) {
            for (int j = 0; j <= 2 * W; ++j) {
              const float c = tapsS[j >= W ? j - W : W - j] * vb[x1 + j];
              const int ci = ib[x1 + j];
              if (better(c, ci, bv, bi)) { bv = c; bi = ci; }
            }
          } else {
            for (int j = 0; j <= 2 * W; ++j) {
              const float c = __ldg(p.band_fwd + (size_t)j * K + x1) * vb[x1 + j];
              const int ci = ib[x1 + j];
              if (better(c, ci, bv, bi)) { bv = c; bi = ci; }
            }
          }
        }
        pr0[q] = valid[q] ? bv : 0.f;
        ix0[q] = bi;
      }
    }

    // delta_t = prior * exp(s (ll_t - max ll_t)), normalised by its sum
    float s2[2] = {0.f, 0.f};
#pragma unroll
    for (int q = 0; q < Q; ++q) {
      de0[q] = pr0[q] * Lc[q];
      de1[q] = pr1 * Lc[q];
      s2[0] += de0[q];
      s2[1] += de1[q];
    }
    group_sum2<WPC>(s2, red, red_par, wig, lane, bar_id);
    const float cn = s2[0] + s2[1];
    const float inv = 1.f / cn;
#pragma unroll
    for (int q = 0; q < Q; ++q) { de0[q] *= inv; de1[q] *= inv; }

    if (t >= t_begin) {
      if (t > 0) {
        int16_t* row = p.bp + (size_t)t * 2 * p.ldbp;
        const int16_t i1 = as_state(ix1, K2);
#pragma unroll
        for (int q = 0; q < Q; ++q) {
          if (valid[q]) {
            const int x = gl + Ge::G * q;
            row[x] = as_state(ix0[q], K2);
            row[p.ldbp + x] = i1;
          }
        }
      }
      if (gl == 0) p.lmr[t] = logf(cn) + scale * m;
    }
    float* msg = nullptr;
    if (t == t_begin - 1 && p.halo_state) msg = p.halo_state + (size_t)s * K2;
    if (t == t_end - 1 && p.end_msg) msg = p.end_msg + (size_t)s * K2;
    if (msg) {
#pragma unroll
      for (int q = 0; q < Q; ++q)
        if (valid[q]) { msg[gl + Ge::G * q] = de0[q]; msg[K + gl + Ge::G * q] = de1[q]; }
    }
    if (p.warm_out) {
      const int j = s + 1;
      const int hn = (p.halo_next_arr && j < p.n_chain) ? p.halo_next_arr[j] : p.halo_next;
      if (t == t_end - hn - 1 && (j < p.n_chain || !p.right_exact)) {
        float* o = p.warm_out + (size_t)j * K2;
#pragma unroll
        for (int q = 0; q < Q; ++q)
          if (valid[q]) { o[gl + Ge::G * q] = de0[q]; o[K + gl + Ge::G * q] = de1[q]; }
      }
    }
  }
}

// words of one rank's record in pmg_viterbi_backtrack_sharded's gathered buffer: link [2K] int32 | last message [2K]
// fp32 | partial sum of lmr (fp64, two words)
__host__ __device__ __forceinline__ int64_t viterbi_record_words(int K) { return 4 * (int64_t)K + 2; }

__device__ __forceinline__ int bp_at(const int16_t* bp, int64_t ldbp, int64_t t, int st, int K) {
  const int d = st >= K;
  const int v = __ldg(bp + (size_t)t * 2 * ldbp + (size_t)d * ldbp + (st - d * K));
  return (unsigned)v < (unsigned)(2 * K) ? v : 0;
}

// maps[c, s] = state at the first core bin of chain c on the best path that ends in state s at its last core bin
__global__ void __launch_bounds__(256) viterbi_maps_kernel(int K, int64_t core_begin, int64_t core_end,
                                                           int64_t chunk_len, const int16_t* bp, int64_t ldbp,
                                                           int* maps) {
  const int c = blockIdx.x;
  const int s0 = blockIdx.y * blockDim.x + threadIdx.x;
  if (s0 >= 2 * K) return;
  const int64_t b = core_begin + (int64_t)c * chunk_len;
  const int64_t e = min(b + chunk_len, core_end);
  int st = s0;
  for (int64_t t = e - 1; t > b; --t) st = bp_at(bp, ldbp, t, st, K);
  maps[(size_t)c * 2 * K + s0] = st;
}

// Chains n_chain-1 .. 0 of a block, from state st at the block's last core bin: path (if given) receives every chain's
// end state (s_{e_{c-1}-1} = bp[b_c, maps[c, s_{e_c-1}]]).  Returns the state at chain 0's first core bin, or with
// through_begin the state one bin before it (one more step through bp[core_begin]).
__device__ int walk_chains(int K, int n_chain, int64_t core_begin, int64_t core_end, int64_t chunk_len,
                           const int16_t* bp, int64_t ldbp, const int* maps, int st, int* path, bool through_begin) {
  for (int c = n_chain - 1; c >= 0; --c) {
    const int64_t b = core_begin + (int64_t)c * chunk_len;
    const int64_t e = min(b + chunk_len, core_end);
    if (path) path[e - 1] = st;
    if (c > 0 || through_begin) st = bp_at(bp, ldbp, b, maps[(size_t)c * 2 * K + st], K);
  }
  return st;
}

// argmax of msg [2K] (ties: smallest index) over the CTA; the result is valid in thread 0
__device__ int block_argmax(const float* msg, int K) {
  __shared__ float sv[8];
  __shared__ int si[8];
  float bv = -INFINITY;
  int bi = INT_MAX;
  for (int i = threadIdx.x; i < 2 * K; i += blockDim.x) {
    const float v = msg[i];
    if (better(v, i, bv, bi)) { bv = v; bi = i; }
  }
  warp_argmax(bv, bi);
  if ((threadIdx.x & 31) == 0) { sv[threadIdx.x >> 5] = bv; si[threadIdx.x >> 5] = bi; }
  __syncthreads();
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
    if (better(sv[w], si[w], bv, bi)) { bv = sv[w]; bi = si[w]; }
  return (unsigned)bi < (unsigned)(2 * K) ? bi : 0;
}

// path[e_c - 1] = end state of every chain: argmax of the last message, then chains from last to first
__global__ void __launch_bounds__(256) viterbi_resolve_kernel(int K, int n_chain, int64_t core_begin,
                                                              int64_t core_end, int64_t chunk_len, const int16_t* bp,
                                                              int64_t ldbp, const int* maps, const float* last_msg,
                                                              int* path) {
  const int st = block_argmax(last_msg, K);
  if (threadIdx.x != 0) return;
  walk_chains(K, n_chain, core_begin, core_end, chunk_len, bp, ldbp, maps, st, path, false);
}

// link[s] = state at bin core_begin - 1 (the left neighbour rank's last core bin) on the best path that ends in state s
// at core_end - 1
__global__ void __launch_bounds__(256) viterbi_link_kernel(int K, int n_chain, int64_t core_begin, int64_t core_end,
                                                           int64_t chunk_len, const int16_t* bp, int64_t ldbp,
                                                           const int* maps, int* link) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= 2 * K) return;
  link[s] = walk_chains(K, n_chain, core_begin, core_end, chunk_len, bp, ldbp, maps, s, nullptr, true);
}

// time-sharded resolve: argmax of the last rank's last message, the links of ranks world-1 .. rank+1 down to this
// rank's end state, then this rank's chains as in viterbi_resolve_kernel
__global__ void __launch_bounds__(256) viterbi_resolve_sharded_kernel(int K, int n_chain, int64_t core_begin,
                                                                      int64_t core_end, int64_t chunk_len,
                                                                      const int16_t* bp, int64_t ldbp,
                                                                      const int* maps, const int* gathered, int world,
                                                                      int rank, int* path) {
  const int64_t rec = viterbi_record_words(K);
  const int* last = gathered + (size_t)(world - 1) * rec;
  int st = block_argmax((const float*)(last + 2 * K), K);
  if (threadIdx.x != 0) return;
  for (int r = world - 1; r > rank; --r) {
    const int v = gathered[(size_t)r * rec + st];
    st = (unsigned)v < (unsigned)(2 * K) ? v : 0;
  }
  walk_chains(K, n_chain, core_begin, core_end, chunk_len, bp, ldbp, maps, st, path, false);
}

// every chain backtracks its own core from its resolved end state
__global__ void __launch_bounds__(128) viterbi_fill_kernel(int K, int n_chain, int64_t core_begin, int64_t core_end,
                                                           int64_t chunk_len, const int16_t* bp, int64_t ldbp,
                                                           int* path) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_chain) return;
  const int64_t b = core_begin + (int64_t)c * chunk_len;
  const int64_t e = min(b + chunk_len, core_end);
  int st = path[e - 1];
  for (int64_t t = e - 1; t > b; --t) {
    st = bp_at(bp, ldbp, t, st, K);
    path[t - 1] = st;
  }
}

template <int Q, int WPC>
static int launch(const Params& p, int n_groups, cudaStream_t st) {
  using Ge = Geo<Q, WPC>;
  const size_t smem = Ge::smem_bytes(p.W);
  if (smem > 227 * 1024) return PMG_ERR_UNSUPPORTED_SHAPE;
  PMG_CUDA_CHECK(cudaFuncSetAttribute(viterbi_fwd_kernel<Q, WPC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
  viterbi_fwd_kernel<Q, WPC><<<cdiv(n_groups, Ge::CPC), 256, smem, st>>>(p);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

// smallest group that covers K with at most 16 bins per thread (pmg_forward's table)
static int dispatch(const Params& p, int n_groups, cudaStream_t st) {
  const int K = p.K;
  if (K <= 32 * 4) return launch<4, 1>(p, n_groups, st);
  if (K <= 32 * 8) return launch<8, 1>(p, n_groups, st);
  if (K <= 32 * 13) return launch<13, 1>(p, n_groups, st);
  if (K <= 32 * 16) return launch<16, 1>(p, n_groups, st);
  if (K <= 64 * 16) return launch<16, 2>(p, n_groups, st);
  if (K <= 128 * 16) return launch<16, 4>(p, n_groups, st);
  if (K <= 256 * 16) return launch<16, 8>(p, n_groups, st);
  return PMG_ERR_UNSUPPORTED_SHAPE;
}

static bool plan_ok(const pmg_scan_plan* plan) {
  return plan && plan->T > 0 && plan->core_begin >= 0 && plan->core_end <= plan->T &&
         plan->core_begin < plan->core_end && plan->chunk_len > 0 && plan->halo >= 0 && plan->n_chain > 0 &&
         (int64_t)plan->n_chain * plan->chunk_len >= plan->core_end - plan->core_begin &&
         (int64_t)(plan->n_chain - 1) * plan->chunk_len < plan->core_end - plan->core_begin;
}

}  // namespace vit
}  // namespace pmg

extern "C" int pmg_viterbi_forward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll,
                                   int64_t ldll, const float* carry_in, const float* warm_in, int64_t warm_stride,
                                   float* warm_out, void* bp, int64_t ldbp, float* lmr, float* halo_state,
                                   float* end_msg, int mode, const int* chain_ids, int n_ids, pmg_stream_t stream) {
  using namespace pmg::vit;
  if (!pmg::vit::plan_ok(plan) || !tr || !ll || !bp || !lmr) return PMG_ERR_BAD_ARG;
  if (tr->K <= 0 || tr->K > 4096 || tr->W < 0 || tr->W > tr->K - 1 + (tr->K == 1)) return PMG_ERR_BAD_ARG;
  if (tr->kind == 0 && (!tr->taps || !tr->inv_z)) return PMG_ERR_BAD_ARG;
  if (tr->kind == 1 && !tr->band_fwd) return PMG_ERR_BAD_ARG;
  if (tr->kind != 0 && tr->kind != 1) return PMG_ERR_BAD_ARG;
  if (mode < 0 || mode > 2 || plan->halo_next < 0) return PMG_ERR_BAD_ARG;
  if (mode == 1 && (!chain_ids || n_ids <= 0)) return PMG_ERR_BAD_ARG;
  if (mode == 2 && !plan->sel_err) return PMG_ERR_BAD_ARG;
  if (mode != 0 && !warm_in) return PMG_ERR_BAD_ARG;   // restarts begin from a snapshot of the carry
  if (ldll < tr->K || ldbp < tr->K) return PMG_ERR_BAD_ARG;
  Params p;
  p.T = plan->T; p.core_begin = plan->core_begin; p.core_end = plan->core_end; p.chunk_len = plan->chunk_len;
  p.n_chain = plan->n_chain; p.halo = plan->halo; p.halo_next = plan->halo_next > 0 ? plan->halo_next : plan->halo;
  p.left_exact = plan->left_exact; p.right_exact = plan->right_exact;
  p.halo_arr = plan->halo_arr; p.halo_next_arr = plan->halo_next_arr;
  p.sel_err = plan->sel_err; p.sel_tol = plan->sel_tol; p.scale = plan->likelihood_scale;
  p.K = tr->K; p.kind = tr->kind; p.W = tr->W; p.taps = tr->taps; p.inv_z = tr->inv_z; p.band_fwd = tr->band_fwd;
  p.M00 = tr->M[0]; p.M01 = tr->M[1]; p.M10 = tr->M[2]; p.M11 = tr->M[3];
  p.ll = ll; p.ldll = ldll; p.carry_in = carry_in; p.warm_in = warm_in; p.warm_stride = warm_stride;
  p.warm_out = warm_out; p.bp = (int16_t*)bp; p.ldbp = ldbp; p.lmr = lmr; p.halo_state = halo_state;
  p.end_msg = end_msg; p.mode = mode; p.chain_ids = chain_ids; p.n_ids = n_ids;
  return dispatch(p, mode == 1 ? n_ids : plan->n_chain, (cudaStream_t)stream);
}

extern "C" int pmg_viterbi_chain_maps(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, int* maps,
                                      pmg_stream_t stream) {
  if (!pmg::vit::plan_ok(plan) || !bp || !maps || K <= 0 || K > 4096 || ldbp < K) return PMG_ERR_BAD_ARG;
  const dim3 grid(plan->n_chain, pmg::cdiv(2 * K, 256));
  pmg::vit::viterbi_maps_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(K, plan->core_begin, plan->core_end,
                                                                       plan->chunk_len, (const int16_t*)bp, ldbp,
                                                                       maps);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_viterbi_backtrack(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp,
                                     const int* maps, const float* last_msg, int* path, pmg_stream_t stream) {
  if (!pmg::vit::plan_ok(plan) || !bp || !maps || !last_msg || !path || K <= 0 || K > 4096 || ldbp < K)
    return PMG_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  pmg::vit::viterbi_resolve_kernel<<<1, 256, 0, st>>>(K, plan->n_chain, plan->core_begin, plan->core_end,
                                                      plan->chunk_len, (const int16_t*)bp, ldbp, maps, last_msg,
                                                      path);
  PMG_LAUNCH_CHECK();
  pmg::vit::viterbi_fill_kernel<<<pmg::cdiv(plan->n_chain, 128), 128, 0, st>>>(
      K, plan->n_chain, plan->core_begin, plan->core_end, plan->chunk_len, (const int16_t*)bp, ldbp, path);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_viterbi_block_link(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, const int* maps,
                                      int* link, pmg_stream_t stream) {
  if (!pmg::vit::plan_ok(plan) || plan->core_begin < 1 || !bp || !maps || !link || K <= 0 || K > 4096 || ldbp < K)
    return PMG_ERR_BAD_ARG;
  pmg::vit::viterbi_link_kernel<<<pmg::cdiv(2 * K, 256), 256, 0, (cudaStream_t)stream>>>(
      K, plan->n_chain, plan->core_begin, plan->core_end, plan->chunk_len, (const int16_t*)bp, ldbp, maps, link);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}

extern "C" int pmg_viterbi_backtrack_sharded(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp,
                                             const int* maps, const int* gathered, int world, int rank, int* path,
                                             pmg_stream_t stream) {
  if (!pmg::vit::plan_ok(plan) || !bp || !maps || !gathered || !path || K <= 0 || K > 4096 || ldbp < K ||
      world < 1 || rank < 0 || rank >= world)
    return PMG_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  pmg::vit::viterbi_resolve_sharded_kernel<<<1, 256, 0, st>>>(K, plan->n_chain, plan->core_begin, plan->core_end,
                                                              plan->chunk_len, (const int16_t*)bp, ldbp, maps,
                                                              gathered, world, rank, path);
  PMG_LAUNCH_CHECK();
  pmg::vit::viterbi_fill_kernel<<<pmg::cdiv(plan->n_chain, 128), 128, 0, st>>>(
      K, plan->n_chain, plan->core_begin, plan->core_end, plan->chunk_len, (const int16_t*)bp, ldbp, path);
  PMG_LAUNCH_CHECK();
  return PMG_OK;
}
