// Chain plan of the time-parallel scans: one definition of the rules every pass over time follows (the filter and
// smoother kernels of pmg_scan.cu, their bulk and compact variants, the lockstep scan of pmg_scan_dense.cu and the
// Viterbi forward pass of pmg_viterbi.cu).
//
//  * validation of a pmg_scan_plan, a pmg_transition and the repair mode (plan_ok, fill_common);
//  * which chain a thread group owns in modes 0, 1 and 2 (chain_range, cta_idle);
//  * per-chain warm-up lengths and where a chain's recursion starts, from which message (halo_own, fwd_start,
//    bwd_start), and where the warm_out message of the next pass is taken (halo_next_of);
//  * the group reductions of a chain's thread group;
//  * the K -> (bins per thread, warps per chain) tiers of the one-chain-per-group kernels (by_tier).
#pragma once
#include <type_traits>

#include "pmg_common.cuh"

namespace pmg {

struct TransDev {
  int K, kind, W;
  const float* taps;
  const float* inv_z;
  const float* band_fwd;
  const float* band_bwd;
  float M00, M01, M10, M11;
};

struct ScanCommon {
  int64_t T, core_begin, core_end, chunk_len;
  int n_chain, halo, left_exact, right_exact;
  int halo_next;            // warm-up length of the NEXT pass: where warm_out messages are taken
  const int* halo_arr;      // optional per-chain warm-up lengths of this pass (overrides halo) ...
  const int* halo_next_arr; // ... and of the next pass (overrides halo_next for chains of this block)
  const float* sel_err;     // mode 2: chain s runs iff !(sel_err[s] <= sel_tol)
  float sel_tol;
  float scale;
  TransDev tr;
  const float* ll;
  int64_t ldll;
  int mode;
  const int* chain_ids;
  int n_ids;
};

// the plan rules documented on pmg_scan_plan (include/pmgplvm_b200.h)
inline bool plan_ok(const pmg_scan_plan* plan) {
  if (!plan || plan->T <= 0 || plan->core_begin < 0 || plan->core_end > plan->T ||
      plan->core_begin >= plan->core_end)
    return false;
  if (plan->chunk_len <= 0 || plan->halo < 0 || plan->halo_next < 0) return false;
  const int64_t n_core = plan->core_end - plan->core_begin;
  // every core bin belongs to a chain, and every chain has at least one
  return (int64_t)plan->n_chain * plan->chunk_len >= n_core && (int64_t)(plan->n_chain - 1) * plan->chunk_len < n_core;
}

// Validates plan, transition and mode of a pass in direction `fwd` and fills c.  A banded transition (kind 1) needs
// the band of the pass's direction.
inline int fill_common(ScanCommon& c, const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll,
                       int64_t ldll, int mode, const int* chain_ids, int n_ids, bool fwd) {
  if (!plan_ok(plan) || !tr || !ll) return PMG_ERR_BAD_ARG;
  if (tr->K <= 0 || tr->W < 0 || tr->W > tr->K - 1 + (tr->K == 1)) return PMG_ERR_BAD_ARG;
  if (tr->kind == 0 && (!tr->taps || !tr->inv_z)) return PMG_ERR_BAD_ARG;
  if (tr->kind == 1 && !(fwd ? tr->band_fwd : tr->band_bwd)) return PMG_ERR_BAD_ARG;
  if (tr->kind != 0 && tr->kind != 1) return PMG_ERR_BAD_ARG;
  if (mode == 1 && (!chain_ids || n_ids <= 0)) return PMG_ERR_BAD_ARG;
  if (mode == 2 && !plan->sel_err) return PMG_ERR_BAD_ARG;
  if (mode < 0 || mode > 2) return PMG_ERR_BAD_ARG;
  if (ldll < tr->K) return PMG_ERR_BAD_ARG;
  c.T = plan->T; c.core_begin = plan->core_begin; c.core_end = plan->core_end;
  c.chunk_len = plan->chunk_len; c.n_chain = plan->n_chain; c.halo = plan->halo;
  c.halo_next = plan->halo_next > 0 ? plan->halo_next : plan->halo;
  c.sel_err = plan->sel_err; c.sel_tol = plan->sel_tol;
  c.halo_arr = plan->halo_arr; c.halo_next_arr = plan->halo_next_arr;
  c.left_exact = plan->left_exact; c.right_exact = plan->right_exact;
  c.scale = plan->likelihood_scale;
  c.tr.K = tr->K; c.tr.kind = tr->kind; c.tr.W = tr->W;
  c.tr.taps = tr->taps; c.tr.inv_z = tr->inv_z; c.tr.band_fwd = tr->band_fwd; c.tr.band_bwd = tr->band_bwd;
  c.tr.M00 = tr->M[0]; c.tr.M01 = tr->M[1]; c.tr.M10 = tr->M[2]; c.tr.M11 = tr->M[3];
  c.ll = ll; c.ldll = ldll; c.mode = mode; c.chain_ids = chain_ids; c.n_ids = n_ids;
  return PMG_OK;
}

// ---- chain selection -------------------------------------------------------
__device__ __forceinline__ int halo_own(const ScanCommon& c, int s) { return c.halo_arr ? c.halo_arr[s] : c.halo; }
// warm-up length chain j will use in the next pass (j outside this block: the neighbour rank's boundary chain)
__device__ __forceinline__ int halo_next_of(const ScanCommon& c, int j) {
  return (c.halo_next_arr && j >= 0 && j < c.n_chain) ? c.halo_next_arr[j] : c.halo_next;
}
// mode 2: true when none of this CTA's chains is selected (the CTA returns before touching shared memory)
__device__ __forceinline__ bool cta_idle(const ScanCommon& c, int chains_per_cta) {
  if (c.mode != 2) return false;
  int any = 0;
  for (int j = threadIdx.x; j < chains_per_cta; j += blockDim.x) {
    const int s = blockIdx.x * chains_per_cta + j;
    if (s < c.n_chain && !(c.sel_err[s] <= c.sel_tol)) any = 1;
  }
  return __syncthreads_or(any) == 0;
}

struct ChainRange {
  int s;
  int64_t t_begin, t_end;
};
// chain of thread group `grp` of this CTA (mode 1: listed chains; mode 2: selected on the device) and its core bins
template <int CPC>
__device__ __forceinline__ bool chain_range(const ScanCommon& c, int grp, ChainRange& r) {
  int idx = blockIdx.x * CPC + grp;
  if (c.mode == 1) {
    if (idx >= c.n_ids) return false;
    r.s = c.chain_ids[idx];
  } else {
    r.s = idx;
  }
  if (r.s < 0 || r.s >= c.n_chain) return false;
  if (c.mode == 2 && c.sel_err[r.s] <= c.sel_tol) return false;   // device-side selection (NaN selects)
  r.t_begin = c.core_begin + (int64_t)r.s * c.chunk_len;
  r.t_end = r.t_begin + c.chunk_len;
  if (r.t_end > c.core_end) r.t_end = c.core_end;
  return r.t_begin < r.t_end;
}

// ---- warm starts -----------------------------------------------------------
// Where a chain's recursion starts and from which message (nullptr: uniform forward, all ones backward).  P is the
// pass's parameter block; its message pointers are read only where the rule needs them.  K: latent bins.
//
// Mode 0 warms up over halo_own bins from p.warm_in; when the warm-up reaches the sequence's exact edge the chain starts
// there exactly instead (forward: bin 0 from p.carry_in; backward: bin T-1 from p.beta_in).  A warm-up longer than
// max_halo bins is cut to max_halo and starts from p.warm_in.
//
// Forward: sets t0, the first bin the recursion visits.  A restart (modes 1, 2) begins at t_begin from p.warm_in (the
// snapshot of the carry), else, with FROM_ALPHA, from the filtered message p.alpha[t0-1], else, at bin 0, from
// p.carry_in.
template <bool FROM_ALPHA, class P>
__device__ __forceinline__ const float* fwd_start(const ScanCommon& c, const ChainRange& cr, const P& p, int64_t& t0,
                                                  int K, int64_t max_halo = INT64_MAX) {
  const float* src = nullptr;
  if (c.mode != 0) {
    t0 = cr.t_begin;
    if (p.warm_in) src = p.warm_in + (size_t)cr.s * p.warm_stride;
    else if constexpr (FROM_ALPHA) {
      if (t0 > 0) src = p.alpha + (size_t)(t0 - 1) * 2 * K;
      else if (p.carry_in) src = p.carry_in;
    } else if (t0 == 0 && p.carry_in) src = p.carry_in;
  } else {
    t0 = cr.t_begin - halo_own(c, cr.s);
    if (t0 <= 0 && c.left_exact && cr.t_begin <= max_halo) {
      t0 = 0;
      src = p.carry_in;
    } else {
      if (t0 < 0) t0 = 0;
      if (cr.t_begin - t0 > max_halo) t0 = cr.t_begin - max_halo;
      if (p.warm_in) src = p.warm_in + (size_t)cr.s * p.warm_stride;
    }
  }
  return src;
}
// Backward: sets t_hi, the first (highest) bin the recursion visits.  A restart begins at the seam bin t_end from
// p.warm_in, else from the next chain's p.beta_end; a chain that ends at bin T-1 starts there from p.beta_in.
// RESTARTS = false compiles the mode-0 rule alone, for a pass that has no restarts (the lockstep scan).
template <bool RESTARTS, class P>
__device__ __forceinline__ const float* bwd_start(const ScanCommon& c, const ChainRange& cr, const P& p, int64_t& t_hi,
                                                  int K, int64_t max_halo = INT64_MAX) {
  const float* init = nullptr;
  if (RESTARTS && c.mode != 0) {
    if (cr.t_end < c.T) {
      t_hi = cr.t_end;
      init = p.warm_in ? p.warm_in + (size_t)cr.s * p.warm_stride : p.beta_end + (size_t)(cr.s + 1) * 2 * K;
    } else { t_hi = c.T - 1; init = p.beta_in; }
  } else {
    t_hi = cr.t_end - 1 + halo_own(c, cr.s);
    if (t_hi >= c.T - 1 && c.right_exact && c.T - cr.t_end <= max_halo) {
      t_hi = c.T - 1;
      init = p.beta_in;
    } else {
      if (t_hi > c.T - 1) t_hi = c.T - 1;
      if (t_hi - (cr.t_end - 1) > max_halo) t_hi = cr.t_end - 1 + max_halo;
      if (p.warm_in) init = p.warm_in + (size_t)cr.s * p.warm_stride;
    }
  }
  return init;
}

// ---- group reductions ------------------------------------------------------
template <int WPC, int NV>
__device__ __forceinline__ void group_sum(float (&v)[NV], float* red, int& red_par, int wig, int lane,
                                          int bar_id) {
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if (WPC > 1) {
    float* r = red + red_par * (WPC * 4);
    if (lane == 0) {
#pragma unroll
      for (int i = 0; i < NV; ++i) r[wig * 4 + i] = v[i];
    }
    named_bar_sync(bar_id, 32 * WPC);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < WPC; ++w) s += r[w * 4 + i];
      v[i] = s;
    }
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

// ---- K tiers -----------------------------------------------------------------
// Calls f(Q, WPC) with compile-time std::integral_constant arguments for the smallest group of WPC warps that covers
// K with at most Q = 16 bins per thread; PMG_ERR_UNSUPPORTED_SHAPE above K = 4096.
template <class F>
int by_tier(int K, F&& f) {
  using Q4 = std::integral_constant<int, 4>;
  using Q8 = std::integral_constant<int, 8>;
  using Q13 = std::integral_constant<int, 13>;
  using Q16 = std::integral_constant<int, 16>;
  using W1 = std::integral_constant<int, 1>;
  if (K <= 32 * 4) return f(Q4{}, W1{});
  if (K <= 32 * 8) return f(Q8{}, W1{});
  if (K <= 32 * 13) return f(Q13{}, W1{});
  if (K <= 32 * 16) return f(Q16{}, W1{});
  if (K <= 64 * 16) return f(Q16{}, std::integral_constant<int, 2>{});
  if (K <= 128 * 16) return f(Q16{}, std::integral_constant<int, 4>{});
  if (K <= 256 * 16) return f(Q16{}, std::integral_constant<int, 8>{});
  return PMG_ERR_UNSUPPORTED_SHAPE;
}

}  // namespace pmg
