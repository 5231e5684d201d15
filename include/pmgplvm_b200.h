/*
 * pmgplvm_b200 — C ABI of the B200-native EM hot path of PoissonGPLVMJump1D.
 *
 * One shared library (libpmgplvm_b200.so), plain pointers and sizes only.  All
 * array pointers are DEVICE pointers owned by the caller (PyTorch allocates
 * them), row-major fp32 unless stated, with explicit leading dimensions in
 * elements.  Every entry point enqueues work on `stream` and returns without a
 * host synchronisation.  Return value: 0 = ok, negative = bad argument
 * (PMG_ERR_*), positive = cudaError_t of a failed runtime call.
 *
 * Each function cites the reference (poor_man_gplvm/...) code it replaces;
 * "SURVEY" ids (E1..D3) are the rows of SURVEY.md section 8(a).
 */
#ifndef PMGPLVM_B200_H
#define PMGPLVM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pmg_stream_t; /* cudaStream_t */

#define PMG_OK 0
#define PMG_ERR_BAD_ARG (-1)
#define PMG_ERR_UNSUPPORTED_SHAPE (-2)
#define PMG_ERR_ALIGNMENT (-3)
#define PMG_ERR_WORKSPACE (-4)

int pmg_version(void);
const char* pmg_error_string(int code);
/* number of SMs of the current device (grid sizing on the host side) */
int pmg_sm_count(void);

/* ------------------------------------------------------------------ E1/E2 --
 * Poisson emission log-likelihood, decoder.py:30-48 vmapped by :60-85, in
 * GEMM form:  ll[t,k] = sum_n y[t,n]*loglam[k,n] - lam_sum[k] - lgam[t],
 * ll[t,k] = -1e20 where ma_latent[k] == 0.
 */

/* loglam[k,n] = ma_neuron[n]*log(tuning[k,n]*dt + 1e-20);
 * lam_sum[k]  = sum_n ma_neuron[n]*(tuning[k,n]*dt + 1e-20).  ma_neuron may be NULL (= ones). */
int pmg_emission_prepare(int K, int N, const float* tuning, const float* ma_neuron, float dt,
                         float* loglam, float* lam_sum, pmg_stream_t stream);

/* lgam[t] = sum_n ma_neuron[n]*lgamma(y[t,n]+1)   (y-only term; constant across EM iterations) */
int pmg_emission_lgamma_rowsum(int64_t T, int N, const float* y, int64_t ldy,
                               const float* ma_neuron, float* lgam, pmg_stream_t stream);

/* Row terms with the full mask surface: ma_neuron is NULL, a vector [N] (ld_mask = 0) or a spatio-temporal
 * mask [T, ld_mask] (decoder.py:291-294).  lgam[t] = sum_n m lgamma(y+1); ysum[t] (optional) = sum_n m y. */
int pmg_emission_row_terms(int64_t T, int N, const float* y, int64_t ldy, const float* ma_neuron,
                           int64_t ld_mask, float* lgam, float* ysum, pmg_stream_t stream);

/* Augmented right-hand operand [rows_out, ldo] (rows >= K zero) for the options the plain GEMM form lacks:
 *  mode 1  [T,N] neuron mask: B[k,:] = [log lam_k | -lam_k], paired with A = [m*y | m]; lam_sum = 0;
 *  mode 2  per-bin dt (decoder.py:73-85): B[k,:] = [ma log(tun_k + 1e-20) | -sum_n ma tun_kn], paired with
 *          A = [y | dt_t]; lam_sum[k] = 1e-20 sum_n ma; the caller adds -log(dt_t) * ysum[t] to lgam[t]. */
int pmg_emission_prepare_aug(int K, int N, const float* tuning, const float* ma_neuron, float dt, int mode,
                             int rows_out, float* out, int64_t ldo, float* lam_sum, pmg_stream_t stream);

/* fp32 operands on CUDA-core tiles: for counts that are not exact in fp16 (non-integer y,
 * decoder.py:37-38) and as the cross-check of the tensor-core kernel below. */
int pmg_emission_poisson(int64_t T, int N, int K, const float* y, int64_t ldy, const float* loglam,
                         const float* lam_sum, const float* lgam, const float* ma_latent,
                         float* ll, int64_t ldll, pmg_stream_t stream);

/* Gaussian observation model (decoder.py:50-57; GaussianGPLVMJump1D / GaussianGPLVM1D, SURVEY 8(f) F2):
 * ll[t,k] = sum_n m * (-(y[t,n] - mu[k,n])^2 / (2 s^2) - log(2 pi s^2) / 2), -1e20 where ma_latent[k] == 0.
 * ma_neuron: NULL, [N] (ld_mask = 0) or [T, ld_mask]. */
int pmg_emission_gaussian(int64_t T, int N, int K, const float* y, int64_t ldy, const float* mu,
                          const float* ma_neuron, int64_t ld_mask, float noise_std, const float* ma_latent,
                          float* ll, int64_t ldll, pmg_stream_t stream);

/* Tensor-core path (tcgen05 kind::f16, TMA-fed, fp32 accumulation in TMEM).
 * y16: fp16 copy of the counts, [T, ld16] with ld16 % 8 == 0 and zero padding; *inexact_count (device)
 *      = number of entries that fp16 does not represent exactly (caller must use the fp32 path if > 0).
 * loglam16: [2, Kpad, ld16] fp16, hi and lo pieces of ma*log(lam) (hi + lo carries 22 bits);
 *      Kpad = ceil(K / BN) * BN with BN = pmg_emission_tile_n(K); padding rows/columns are zero. */
int pmg_counts_to_f16(int64_t T, int N, const float* y, int64_t ldy, void* y16, int64_t ld16,
                      int* inexact_count, pmg_stream_t stream);

/* The two passes above fused (one read of the counts): fp16 copy [T, ld16] with an optional column of ones at
 * index N (ones_col; the statistics GEMM then also returns sum_t gamma) and zero padding up to ld16, the exactness
 * counter, lgam[t] = sum_n m_n lgamma(y[t,n]+1) (reference decoder.py:40) and optionally ysum[t] = sum_n m_n y[t,n].
 * ma_neuron: NULL or a vector [N]. */
int pmg_counts_prepare(int64_t T, int N, const float* y, int64_t ldy, const float* ma_neuron, void* y16,
                       int64_t ld16, int ones_col, int* inexact_count, float* lgam, float* ysum,
                       pmg_stream_t stream);
/* Shuffle tests (reference test.py:22-23, np.roll per neuron): the fp16 operand and lgam of pmg_counts_prepare
 * (ones_col = 0) for n_shift circular shuffles stacked along time,
 *   y16[b*T + t, n] = y[(t - shifts[b*N + n]) mod T, n],   lgam[b*T + t] = sum_n m_n lgamma(y16[b*T + t, n] + 1),
 * bit-identical to pmg_counts_prepare run on each rolled fp32 matrix.  Source: the fp16-exact counts in NEURON-MAJOR
 * layout yT16 [N, ld_src] (a neuron's shifted window is contiguous).  Out: y16 [n_shift*T, ld16] fp16 (zero padding
 * from column N), lgam [n_shift*T].  shifts: device int32 [n_shift, N], each in [0, T).  ma_neuron: NULL or [N].
 * No exactness counter: a circular shift does not change the set of values of a column. */
int pmg_counts_prepare_shifted(int64_t T, int N, int n_shift, const void* yT16, int64_t ld_src, const int* shifts,
                               const float* ma_neuron, void* y16, int64_t ld16, float* lgam, pmg_stream_t stream);
int pmg_emission_tile_n(int K);
int pmg_emission_prepare_f16(int K, int N, const float* tuning, const float* ma_neuron, float dt, int Kpad,
                             int64_t ld16, void* loglam16, float* lam_sum, pmg_stream_t stream);
int pmg_emission_poisson_f16(int64_t T, int N, int K, const void* y16, int64_t ld16, const void* loglam16,
                             int Kpad, const float* lam_sum, const float* lgam, const float* ma_latent,
                             float* ll, int64_t ldll, pmg_stream_t stream);

/* -------------------------------------------------------------------- E3 --
 * Naive-Bayes normalisation, decoder.py:88-102: lml_t = logsumexp_k ll[t,:],
 * log_post = ll - lml_t.  log_post may alias ll.
 */
int pmg_naive_bayes_normalize(int64_t T, int K, const float* ll, int64_t ldll, float* log_post,
                              int64_t ldp, float* lml_t, pmg_stream_t stream);
/* same, also writing post = exp(log_post) ([T, ldp]; core.py:517) in the one pass over the rows */
int pmg_naive_bayes_posterior(int64_t T, int K, const float* ll, int64_t ldll, float* log_post, float* post,
                              int64_t ldp, float* lml_t, pmg_stream_t stream);
/* lml_t alone (a read-only pass over ll), bit-identical to the lml_t of the two entries above */
int pmg_naive_bayes_lml(int64_t T, int K, const float* ll, int64_t ldll, float* lml_t, pmg_stream_t stream);

/* ------------------------------------------------------------- F1/F2, S1-S3 --
 * Forward filter (decoder.py:151-198) and backward smoother (decoder.py:200-332)
 * in linear space (SURVEY Appendix A), parallel in time over `n_chain`
 * contiguous chunks of `chunk_len` bins; a chain warms up over `halo` bins
 * from the uniform carry and records its warmed-up state so that
 * pmg_seam_check can verify it against the neighbouring chain's true state.
 */
typedef struct pmg_transition {
  int K;              /* latent bins */
  int kind;           /* 0 = Toeplitz RBF: P0[x,x'] = taps[|x-x'|]*inv_z[x];  1 = banded/dense general */
  int W;              /* band half width: P0[x,x'] == 0 for |x-x'| > W */
  const float* taps;  /* kind 0: [W+1] */
  const float* inv_z; /* kind 0: [K] */
  const float* band_fwd; /* kind 1: [2W+1, K]: band_fwd[j,x'] = P0[x'-W+j, x'] (0 outside) */
  const float* band_bwd; /* kind 1: [2W+1, K]: band_bwd[j,x ] = P0[x, x-W+j]  (0 outside) */
  float M[4];         /* dynamics transition M[d,d'] row-major, (from, to) */
} pmg_transition;

typedef struct pmg_scan_plan {
  int64_t T;          /* bins held locally (including any halo bins fetched from neighbours) */
  int64_t core_begin; /* outputs are produced for bins [core_begin, core_end) */
  int64_t core_end;
  int64_t chunk_len;  /* bins per chain */
  int n_chain;        /* ceil((core_end-core_begin)/chunk_len) */
  int halo;           /* warm-up bins */
  int left_exact;     /* bin 0 is the true start of the sequence (or carry_in is exact) */
  int right_exact;    /* bin T-1 is the true end of the sequence (or beta_in is exact) */
  float likelihood_scale;
  int halo_next;      /* warm-up length of the NEXT pass (where warm_out messages are taken); 0 = halo */
  float sel_tol;      /* mode 2: chain s is re-run iff !(sel_err[s] <= sel_tol) */
  const float* sel_err; /* mode 2: device array [n_chain] of seam errors (pmg_seam_check_fix) */
  const int* halo_arr;      /* optional device int32 [n_chain]: per-chain warm-up lengths of this pass (overrides halo) */
  const int* halo_next_arr; /* optional device int32 [n_chain]: per-chain warm-up lengths of the next pass */
} pmg_scan_plan;

/* mode 0: all chains, warm-up from the uniform carry (left-most chain exact if left_exact).
 * mode 1: relay — run only chains listed in chain_ids[n_ids] (device int32) starting
 *         from the exact carry alpha[t_begin-1].
 * mode 2: like mode 1 with the selection made on the device: every chain s with !(plan->sel_err[s] <=
 *         plan->sel_tol) restarts from its snapshot (warm_in), the others return at once.  Together with
 *         pmg_seam_check_fix this repairs failed seams without a host round trip.
 * alpha:   [T, 2, K] (ld = 2*ldk), lmr: [T] = log c_t + s*max_k ll[t,k]
 * carry_in: [2,K] or NULL (uniform);   halo_state: [n_chain, 2, K] warmed-up state at t_begin-1.
 * warm_in:  message a warm-up starts from: one [2,K] vector (warm_stride 0, e.g. the stationary
 *           distribution of the prior chain) or one per chain (warm_stride 2K: the previous EM
 *           iteration's message at that bin); NULL = uniform.  warm_out: [n_chain,2,K] or NULL,
 *           receives the message at each chain's warm-up start for the next pass (forward: chain c writes
 *           slot c+1; backward: chain c writes slot c-1).  Time-sharded blocks: when right_exact == 0 the
 *           forward pass also writes slot n_chain (the right neighbour's first chain) and when left_exact == 0
 *           the backward pass also writes slot -1 (the left neighbour's last chain): the caller provides the
 *           extra slot (forward: [n_chain+1,2,K]; backward: pass a pointer to slot 1 of [n_chain+1,2,K]). */
int pmg_forward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                float* alpha, float* lmr, float* halo_state, int mode,
                const int* chain_ids, int n_ids, pmg_stream_t stream);

/* gamma:      [T, 2, K] or NULL; gamma_lat: [T, K] or NULL (sum over dynamics); dyn_marg: [T,2] or NULL
 * gamma16:    [2, T, ldg] fp16 or NULL: hi/lo pieces of gamma_lat (ldg % 8 == 0; padding columns are not
 *             written: zero them once) for pmg_atb_f16
 * r_out:      [T, 2, K] or NULL (r[t] = L_t*beta_t/c_t, the right factor of the transition counts)
 * tw_partial: [n_chain, K] or NULL (per-chain sum_t gamma_lat)
 * beta_in:    [2,K] or NULL (ones);  beta_halo / beta_end: [n_chain, 2, K]. */
int pmg_backward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                 const float* alpha, const float* beta_in, const float* warm_in, int64_t warm_stride,
                 float* warm_out, float* gamma, float* gamma_lat,
                 void* gamma16, int64_t ldg, float* dyn_marg, float* r_out, float* tw_partial, float* beta_halo, float* beta_end,
                 int mode, const int* chain_ids, int n_ids, pmg_stream_t stream);

/* pmg_backward that writes the operands of the transition-count GEMM (decoder.py:215-221, SURVEY S4) directly as
 * bf16 hi/lo pieces instead of the fp32 r_out -- no separate pmg_split_bf16 passes over two [T,2K] arrays:
 *   row t   of xa_hi / xa_lo [T, ld_x] = alpha_t [2K]           (hi = bf16(v), lo = bf16(v - hi))
 *   row t+1 of xr_hi / xr_lo [T, ld_x] = r_{t+1} / z_t [2K]
 * for the core bins t (rows nobody writes are left untouched).  ld_x >= 2K, ld_x % 8 == 0, 16-byte aligned pointers.
 * Supported where pmg_backward runs its bulk kernel (pmg_backward_xi16_supported: Toeplitz kernel with W <= 10,
 * K % 8 == 0, K <= 512, likelihood_scale > 0); PMG_ERR_UNSUPPORTED_SHAPE otherwise.  Feed the pieces to
 * pmg_atb_bf16x2_pieces. */
int pmg_backward_xi16_supported(const pmg_transition* tr, float likelihood_scale);
int pmg_backward_xi16(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                      const float* alpha, const float* beta_in, const float* warm_in, int64_t warm_stride,
                      float* warm_out, float* gamma, float* gamma_lat, void* gamma16, int64_t ldg, float* dyn_marg,
                      void* xa_hi, void* xa_lo, void* xr_hi, void* xr_lo, int64_t ld_x, float* tw_partial,
                      float* beta_halo, float* beta_end, int mode, const int* chain_ids, int n_ids,
                      pmg_stream_t stream);

/* err[i] = max relative difference between est[i,:]/sum(est[i,:]) and truth[i,:]/sum(truth[i,:]) over entries
 * whose normalised value is > floor (messages are defined up to a positive scale: every step of both passes
 * renormalises).  est/truth are [n, len] with row strides in elements (truth rows may live inside alpha). */
int pmg_seam_check(int n, int len, const float* est, int64_t ld_est, const float* truth,
                   int64_t ld_truth, float floor_val, float* err, pmg_stream_t stream);
/* Same check; seams with !(err <= tol) add 1 to *counter (device float, may be NULL) and, with fix != 0, have
 * their estimate row overwritten by the truth row -- the snapshot a mode-2 restart of that chain starts from. */
int pmg_seam_check_fix(int n, int len, float* est, int64_t ld_est, const float* truth, int64_t ld_truth,
                       float floor_val, float tol, int fix, float* err, float* counter, pmg_stream_t stream);
/* EM-iteration fast path of the two passes ("compact" filtered posterior).  The filtered jump-state
 * message is a scalar multiple of the likelihood factor, alpha_t[1,x] = a1s_t * exp2(s*log2e*(ll[t,x] -
 * max_x ll[t,:])), so the forward pass stores ax[T, ldax] with columns 0..K-1 = alpha_t[0,:], column K =
 * a1s_t, column K+1 = lmr_t (ldax >= K+4, ldax % 4 == 0) and the backward pass rebuilds alpha_t[1,:] from
 * the ll row; it emits only what an EM iteration consumes (gamma16; sum_t gamma comes out of the statistics
 * GEMM through a column of ones appended to the counts) plus the seam messages.
 * Supported: kind 0 (Toeplitz), W <= 10, K % 8 == 0, K <= 496, M[0] > 0, likelihood_scale > 0
 * (pmg_scan_compact_supported); everything else uses pmg_forward / pmg_backward.
 * fwd_end: [n_chain,2,K] true message at the last bin of each chain; first_out: [2,K] true message at
 * core_begin; mode 1 restarts the listed chains from warm_in (a snapshot of their carry). */
int pmg_scan_compact_supported(const pmg_transition* tr, float likelihood_scale);
int pmg_forward_compact(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                        const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                        float* ax, int64_t ldax, float* halo_state, float* fwd_end, float* first_out,
                        int mode, const int* chain_ids, int n_ids, pmg_stream_t stream);
int pmg_backward_compact(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                         const float* ax, int64_t ldax, const float* beta_in, const float* warm_in,
                         int64_t warm_stride, float* warm_out, void* gamma16, int64_t ldg,
                         float* beta_halo, float* beta_end, int mode, const int* chain_ids, int n_ids,
                         pmg_stream_t stream);

/* Viterbi decoding (beyond the reference, which returns marginals only): the most probable joint path of the
 * (dynamics, latent) chain, s = d*K + x, transition M[d,d'] P_{d'}[x,x'] with P_1 = 1/K.  Bin 0's prior is the one
 * pmg_forward forms from carry_in (the start is marginalised), every later bin takes the max over predecessors;
 * exact ties go to the smallest flat index d*K + x.  Time-parallel over the chains of pmg_forward.
 *
 * pmg_viterbi_forward: plan, transition (kind 0 or 1, any K <= 4096), warm starts (carry_in, warm_in, warm_stride,
 *   warm_out), mode 0/1/2 and chain_ids exactly as pmg_forward; modes 1 and 2 need warm_in (the carry snapshots).
 *   Messages are normalised by their sum every bin, as in the filter, so pmg_seam_check_fix applies to them.
 *   bp:       int16 [T, 2, ldbp] (ldbp >= K): bp[t, d', x'] = flat predecessor state of (d', x') at bin t, written
 *             for the core bins t > 0 (row 0 is unused);
 *   lmr:      [T] = log(sum of the unnormalised message) + s*max_k ll[t,k] at the core bins, so that
 *             log max_path p(path, y) = sum_t lmr[t] + log max(message at the last bin);
 *   halo_state: [n_chain, 2, K] or NULL, the warmed-up message at t_begin-1 (the seam estimate);
 *   end_msg:  [n_chain, 2, K] or NULL, the message at each chain's last core bin (the seam truth of the next chain;
 *             the last one is the message pmg_viterbi_backtrack starts from). */
int pmg_viterbi_forward(const pmg_scan_plan* plan, const pmg_transition* tr, const float* ll, int64_t ldll,
                        const float* carry_in, const float* warm_in, int64_t warm_stride, float* warm_out,
                        void* bp, int64_t ldbp, float* lmr, float* halo_state, float* end_msg, int mode,
                        const int* chain_ids, int n_ids, pmg_stream_t stream);
/* maps: device int32 [n_chain, 2K]; maps[c, s] = the state at chain c's first core bin on the best path that ends
 * in state s at its last core bin (2K threads per chain follow bp through the chain's core). */
int pmg_viterbi_chain_maps(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, int* maps,
                           pmg_stream_t stream);
/* path: device int32 [T] (core bins written), the flat states d*K + x of the MAP path.  Two launches: one CTA takes
 * the argmax of last_msg [2K] and resolves every chain's end state from the last chain to the first
 * (s_{b_c} = maps[c, s_{e_c-1}], s_{e_{c-1}-1} = bp[b_c, s_{b_c}]), then every chain fills its core. */
int pmg_viterbi_backtrack(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, const int* maps,
                          const float* last_msg, int* path, pmg_stream_t stream);
/* Time-sharded Viterbi: each rank holds bp for its own core bins (plus halo rows), so the single-device resolve of
 * pmg_viterbi_backtrack, which walks every chain of the recording, is split in two.
 * pmg_viterbi_block_link: link, device int32 [2K]; link[s] = the state at bin core_begin - 1 (the left neighbour's last
 *   core bin) on the best path that ends in state s at core_end - 1.  2K threads each walk the chains from last to
 *   first (the resolve loop of pmg_viterbi_backtrack, ~2 n_chain dependent loads) and take one more step through
 *   bp[core_begin]; needs core_begin >= 1 (a rank with a left neighbour).
 * pmg_viterbi_backtrack_sharded: replaces pmg_viterbi_backtrack on a rank of a time-sharded decode.  gathered: device
 *   int32 [world][4K + 2], every rank's record in rank order: link [2K] int32 | its last message [2K] fp32 | the fp64
 *   partial sum of its lmr (two words; not read here).  One CTA takes the argmax of the last rank's message (ties:
 *   smallest index), follows the links of ranks world-1 .. rank+1 to this rank's end state and resolves the chain end
 *   states; then every chain fills its core, as in pmg_viterbi_backtrack.  No other collective, no host round trip. */
int pmg_viterbi_block_link(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, const int* maps, int* link,
                           pmg_stream_t stream);
int pmg_viterbi_backtrack_sharded(const pmg_scan_plan* plan, int K, const void* bp, int64_t ldbp, const int* maps,
                                  const int* gathered, int world, int rank, int* path, pmg_stream_t stream);

/* Dense / wide-band move kernels (gp_kernel.py:61-66 custom_transition_kernel; :14-20 with a large
 * movement_variance; BASELINE configs[4]) on the tensor cores: all chains advance in LOCKSTEP, so the n_chain
 * mat-vecs of one time step are one [n_chain x K] . [K x K] GEMM (tcgen05 kind::f16, both operands as two fp16
 * pieces under exact power-of-two scales, three products, fp32 accumulation), followed by a per-chain row kernel
 * (likelihood factor, rank-1 jump term, normaliser, outputs, seam / warm-start messages).  Same chain, warm-up
 * and output conventions as pmg_forward / pmg_backward, mode 0 only (repairs go through those).
 * P16: device fp16 [2 directions][2 pieces][Kn][Kk] (256-byte aligned) with, for the row-normalised move matrix P0,
 *      direction 0 (forward):  B[x', x] = 2^14 * P0[x, x'],  direction 1 (backward): B[x, x'] = 2^14 * P0[x, x'],
 *      piece 0 = fp16(B), piece 1 = fp16(B - piece 0), zero padding; (Kk, Kn) from pmg_dense_scan_geometry.
 * kb_ranges: HOST int32 [2 directions][n_ntiles][2] = first / one-past-last 64-column block that holds a non-zero
 *      of rows [i*BN, (i+1)*BN) of B (band structure; NULL = all blocks).
 * halo_max: upper bound of plan->halo_arr (ignored without per-chain warm-ups); a pass is halo_max + chunk_len steps.
 * workspace: pmg_dense_scan_workspace_bytes(n_chain, K) bytes, 256-byte aligned. */
int pmg_dense_scan_geometry(int K, int* Kk, int* Kn, int* BN, int* n_ntiles);
int64_t pmg_dense_scan_workspace_bytes(int n_chain, int K);
int pmg_forward_dense(const pmg_scan_plan* plan, const pmg_transition* tr, const void* P16, const int* kb_ranges,
                      int halo_max, const float* ll, int64_t ldll, const float* carry_in, const float* warm_in,
                      int64_t warm_stride, float* warm_out, float* alpha, float* lmr, float* halo_state,
                      void* workspace, int64_t workspace_bytes, pmg_stream_t stream);
int pmg_backward_dense(const pmg_scan_plan* plan, const pmg_transition* tr, const void* P16, const int* kb_ranges,
                       int halo_max, const float* ll, int64_t ldll, const float* alpha, const float* beta_in,
                       const float* warm_in, int64_t warm_stride, float* warm_out, float* gamma, float* gamma_lat,
                       void* gamma16, int64_t ldg, float* dyn_marg, float* r_out, float* tw_partial,
                       float* beta_halo, float* beta_end, void* workspace, int64_t workspace_bytes,
                       pmg_stream_t stream);

/* Boundary messages of a time-sharded forward pass (SURVEY 8(e); the reference is single-device), one small kernel
 * on each side of the exchange instead of ~20 tensor ops.  out [8K] = [to_left: first (2K) | unused (2K) |
 * to_right: last (2K) | warm (2K)] with `warm` = this pass's message at the bin in front of the right neighbour's next
 * warm-up: warm_mode 0 zeros, 1 = warm_src [2K], 2 = built from a compact row (ax_row [K+4], ll_row [K]).
 * unpack: from_left [4K] (the left rank's to_right) -> fwd_end0 [2K] (seam truth), fwarm0 [2K] (warm start, may be
 * NULL); from_right [4K] (the right rank's to_left) -> the row behind this block: alpha_stop [2K], or with compact != 0
 * ax_stop [K+4] (alpha[0,:] and the scalar a1s for ll_stop [K]).  NULL inputs are skipped. */
int pmg_boundary_pack_fwd(int K, const float* first, const float* last, int warm_mode, const float* warm_src,
                          const float* ax_row, const float* ll_row, float likelihood_scale, float* out,
                          pmg_stream_t stream);
int pmg_boundary_unpack_fwd(int K, const float* from_left, const float* from_right, float* fwd_end0, float* fwarm0,
                            int compact, float* ax_stop, const float* ll_stop, float likelihood_scale,
                            float* alpha_stop, pmg_stream_t stream);

/* dst[0] = sum_{i<n} src[i*stride], accumulated in fp64 in a fixed order (the log marginal of a pass is the sum of the
 * one-step predictive log marginals, decoder.py:170,186).  workspace: pmg_strided_sum_workspace_bytes() bytes,
 * 8-byte aligned, zeroed ONCE by the caller (the kernel re-arms it); one call at a time per workspace. */
int64_t pmg_strided_sum_workspace_bytes(void);
int pmg_strided_sum(int64_t n, const float* src, int64_t stride, float* dst, void* workspace, pmg_stream_t stream);

/* ------------------------------------------------------------------ M1, S4 --
 * C[m,n] = sum_t A[t,m]*B[t,n]  (time is the reduction axis).  Used for the
 * sufficient statistics (fit_tuning_helper.py:28-42: A = gamma_lat, B = y) and
 * for the transition counts (decoder.py:215-221 via SURVEY S4: A = alpha, B = r).
 * workspace: pmg_atb_workspace_bytes(...) bytes, or NULL when that returns 0.
 */
int64_t pmg_atb_workspace_bytes(int64_t T, int M, int N, int impl);
int pmg_atb(int64_t T, int M, int N, const float* A, int64_t lda, const float* B, int64_t ldb,
            float* C, int64_t ldc, void* workspace, int64_t workspace_bytes, int impl,
            pmg_stream_t stream);

/* Tensor-core time reduction for the sufficient statistics (tcgen05 kind::f16, both operands
 * MN-major, split over time, fixed-order fp64 reduction of the splits):
 *   yw[k,n] = sum_t (g16[0,t,k] + g16[1,t,k]) * y16[t,n]
 * g16: [2, T, ldg] fp16 pieces of the posterior (pmg_split_f16 or pmg_backward's gamma16);
 * y16: [T, ldy16] fp16 counts (pmg_counts_to_f16). */
int pmg_split_f16(int64_t T, int K, const float* src, int64_t lds, void* dst16, int64_t ld16, pmg_stream_t stream);
int64_t pmg_atb_f16_workspace_bytes(int64_t T, int K, int N);
int pmg_atb_f16(int64_t T, int K, int N, const void* g16, int64_t ldg, const void* y16, int64_t ldy16,
                float* yw, void* workspace, int64_t workspace_bytes, pmg_stream_t stream);

/* Time reduction with BOTH operands split into two bf16 pieces ([2, T, ld], hi then lo; 16 significant bits,
 * fp32 exponent range): out[k,n] = sum_t G[t,k] * Y[t,n] as three tensor-core products (hi*hi + hi*lo + lo*hi)
 * accumulated in fp32; relative error ~2^-16 per term.  Used for the transition counts (SURVEY S4,
 * decoder.py:215-221: G = alpha [T,2K], Y = r shifted by one bin).  ld % 8 == 0, 16-byte aligned pointers;
 * workspace: pmg_atb_f16_workspace_bytes(T, K, N). */
int pmg_split_bf16(int64_t T, int K, const float* src, int64_t lds, void* dst16, int64_t ld16, pmg_stream_t stream);
int pmg_atb_bf16x2(int64_t T, int K, int N, const void* g16, int64_t ldg, const void* y16, int64_t ldy16,
                   float* out, void* workspace, int64_t workspace_bytes, pmg_stream_t stream);

/* pmg_atb_bf16x2 with every piece behind its own pointer (T rows each; ldg / ldy16 per operand): the pieces written
 * by pmg_backward_xi16 are used in place, at a row offset (alpha rows [t0, t1) against r rows [t0+1, t1+1)). */
int pmg_atb_bf16x2_pieces(int64_t T, int K, int N, const void* g_hi, const void* g_lo, int64_t ldg,
                          const void* y_hi, const void* y_lo, int64_t ldy16, float* out, void* workspace,
                          int64_t workspace_bytes, pmg_stream_t stream);

/* log_acc[d,d',x,x'] = logM[d,d'] + logP_{d'}[x,x'] + log G[(d,x),(d',x')]   (G = alpha^T r, [2K,2K]):
 * decoder.py:221's accumulator; using the analytic log kernel keeps deep tails finite.
 * logP: device [2,K,K]; logM: HOST float[4] row-major (from, to). */
int pmg_xi_finalize(int K, const float* G, const float* logP, const float* logM,
                    float* log_acc /*[2,2,K,K]*/, pmg_stream_t stream);

/* -------------------------------------------------------------------- M2/M3 --
 * Adam M-step, fit_tuning_helper.py:124-196 on the objective :63-81 with the
 * softplus link :19-25.  One cooperative persistent kernel; CTA per neuron tile.
 * W, mu, nu: [B,N] in/out; count: device int32 in/out (optax count);
 * loss_hist/err_hist: [maxiter] out (zero beyond n_iter); n_iter_out: device int32;
 * final: device float[2] = (final_loss, final_error); tuning_out: [K,N] = softplus(Phi W_final).
 * workspace: pmg_mstep_workspace_bytes(...) bytes, zero-initialised by the callee.
 */
int64_t pmg_mstep_workspace_bytes(int K, int B, int N, int maxiter);
int pmg_mstep_adam(int K, int B, int N, const float* Phi, const float* yw, const float* tw,
                   float prior_std, float lr, float b1, float b2, float eps, int maxiter, float tol,
                   int min_iters, float* W, float* mu, float* nu, int* count, float* loss_hist,
                   float* err_hist, int* n_iter_out, float* final_out, float* tuning_out,
                   void* workspace, int64_t workspace_bytes, pmg_stream_t stream);

/* Same with strided statistics: yw[k,n] at yw[k*ldyw + n], tw[k] at tw[k*tw_stride] -- the [K, N+1] output of
 * pmg_atb_f16 on counts with a ones column is consumed in place (yw = out, ldyw = N+1, tw = out + N, stride N+1). */
int pmg_mstep_adam_ld(int K, int B, int N, const float* Phi, const float* yw, int64_t ldyw, const float* tw,
                      int64_t tw_stride, float prior_std, float lr, float b1, float b2, float eps, int maxiter,
                      float tol, int min_iters, float* W, float* mu, float* nu, int* count, float* loss_hist,
                      float* err_hist, int* n_iter_out, float* final_out, float* tuning_out,
                      void* workspace, int64_t workspace_bytes, pmg_stream_t stream);

/* tuning[k,n] = softplus(sum_b Phi[k,b]*W[b,n])   (fit_tuning_helper.py:11-25) */
int pmg_tuning_softplus(int K, int B, int N, const float* Phi, const float* W, float* tuning,
                        pmg_stream_t stream);

/* ---------------------------------------------------------------------- D2 --
 * Initial latent posterior, core.py:571-583, with jax.random's bit stream (threefry2x32, jax 0.4.26 defaults):
 * rows [t_offset, t_offset+T) of uniform(key, (T_total, K)) * random_scale, row-normalised.  Any of the outputs
 * may be NULL: post [T, ldp] fp32, logpost [T, ldl] fp32, g16 = fp16 hi/lo pieces (hi at g16, lo at
 * g16 + piece_stride halves, row stride ldg), tw [K] fp64 = column sums of post (zeroed by the callee).
 * Requires T_total*K < 2^32 (one counter block of the reference's generator). */
int pmg_threefry_posterior_init(int64_t T, int K, int64_t t_offset, int64_t T_total, uint32_t key0, uint32_t key1,
                                float random_scale, float* post, int64_t ldp, float* logpost, int64_t ldl,
                                void* g16, int64_t ldg, int64_t piece_stride, double* tw, pmg_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PMGPLVM_B200_H */
