"""PoissonGPLVMJump1D — drop-in for the reference class of the same name.

Host logic of reference ``poor_man_gplvm/core.py``: ``AbstractGPLVMJump1D``
(:376-733) and ``PoissonGPLVMJump1D`` (:746-849).  Same constructor, method
names, keyword arguments and result-dictionary keys; the numerics run in the
hand-written sm_100a kernels behind ``libpmgplvm_b200.so`` (no JAX, no CPU
fallback).  Arrays come back as NumPy arrays (pass ``return_device=True`` to
``fit_em`` / ``decode_latent*`` to keep T-sized results on the GPU as torch
tensors and skip the device->host copies).
"""
from __future__ import annotations

import contextlib
import functools
import os
import time

import numpy as np
import torch

from . import gp_kernel as gpk
from . import hostio
from . import jaxprng
from . import ops
from . import estep
from . import viterbi
from .estep import EStep
from .shard import TimeShard


def _unwrap_tsd(y):
    """pynapple TsdFrame duck-typing (reference core.py:459-461): returns (values, times or None)."""
    if hasattr(y, "d") and hasattr(y, "t") and not isinstance(y, (np.ndarray, torch.Tensor)):
        return y.d, y.t
    return y, None


def _rewrap_tsd(arr, t_l):
    if t_l is None:
        return arr
    try:
        import pynapple as nap   # optional; only when the caller handed us a TsdFrame
        return nap.TsdFrame(d=arr, t=t_l)
    except Exception:
        return arr


def _rewrap_tsd_1d(arr, t_l):
    if t_l is None:
        return arr
    try:
        import pynapple as nap   # optional; only when the caller handed us a TsdFrame or t_l
        return nap.Tsd(t=t_l, d=arr)
    except Exception:
        return arr


class _Timing:
    """Optional wall-clock breakdown of fit_em (PMG_TIMING=1): synchronises at every mark."""

    def __init__(self):
        self.on = bool(os.environ.get("PMG_TIMING"))
        self.per_iter = os.environ.get("PMG_TIMING") in ("2", "3")
        self.nosync = os.environ.get("PMG_TIMING") == "3"       # host-side marks only (no perturbation)
        self.iters = []
        self.t = time.perf_counter()
        self.marks = []

    def mark(self, name):
        if self.on:
            if not self.nosync:
                torch.cuda.synchronize()
            now = time.perf_counter()
            self.marks.append((name, now - self.t))
            self.t = now

    def iteration(self):
        """PMG_TIMING=2: wall time of every EM iteration (synchronised; perturbs the loop)."""
        if self.per_iter:
            if not self.nosync:
                torch.cuda.synchronize()
            now = time.perf_counter()
            self.iters.append(now - self.t_it)
            self.t_it = now

    def report(self):
        if self.on:
            print("fit_em timing: " + ", ".join("%s %.3fs" % m for m in self.marks), flush=True)
        if self.per_iter:
            print("fit_em iterations (ms): " + " ".join("%.1f" % (x * 1e3) for x in self.iters), flush=True)


def _seed_from_key(key):
    """seed for the NumPy generators of sample* (jax.random.poisson / choice are not restated)"""
    if key is None:
        return 0
    a = np.asarray(key).astype(np.uint64).ravel()
    return int(a[-1]) if a.size else 0


# above this many entries the initial posterior is drawn on the device (pmg_threefry_posterior_init)
_HOST_PRNG_MAX = 1 << 22


def compute_transition_posterior_prob(log_acc):
    """reference decoder.py:334-375 on a torch tensor [2,2,K,K] -> dict of 12 tensors."""
    lse = torch.logsumexp
    log_joint_full = log_acc - lse(log_acc.reshape(-1), 0)
    log_joint_latent = lse(log_joint_full, dim=(0, 1))
    log_joint_dynamics = lse(log_joint_full, dim=(2, 3))
    log_transition_latent = log_joint_latent - lse(log_joint_latent, dim=1, keepdim=True)
    log_transition_dynamics = log_joint_dynamics - lse(log_joint_dynamics, dim=1, keepdim=True)
    log_transition_full = log_joint_full - lse(log_joint_full, dim=(1, 3), keepdim=True)
    res = {'p_joint_full': torch.exp(log_joint_full),
           'p_joint_latent': torch.exp(log_joint_latent),
           'p_joint_dynamics': torch.exp(log_joint_dynamics),
           'p_transition_full': torch.exp(log_transition_full),
           'p_transition_latent': torch.exp(log_transition_latent),
           'p_transition_dynamics': torch.exp(log_transition_dynamics),
           'log_joint_full': log_joint_full,
           'log_joint_latent': log_joint_latent,
           'log_joint_dynamics': log_joint_dynamics,
           'log_transition_full': log_transition_full,
           'log_transition_latent': log_transition_latent,
           'log_transition_dynamics': log_transition_dynamics}
    return res


def _on_device(fn):
    """Runs a public method with the model's device current: every kernel launches on the current device's current
    stream, so a model built with ``device='cuda:1'`` must not depend on the caller having selected that device."""
    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        dev = self.device if (self._device is not None or torch.cuda.is_available()) else None
        guard = torch.cuda.device(dev) if (dev is not None and dev.type == "cuda") else contextlib.nullcontext()
        with guard:
            return fn(self, *args, **kwargs)
    return wrapper


class EMLoop:
    """Device-resident state of one EM run (reference core.py:640-676): the posterior over latent bins,
    the GLM weights with their Adam state, and the E-step buffers.  ``iteration`` is the loop body of
    ``fit_em``: statistics -> Adam M-step -> tuning -> E-step."""

    def __init__(self, model, y_dev, op, ma_n, ma_l, likelihood_scale, tuning_basis, log_posterior_init, prior_std,
                 step_size=0.01, maxiter=1000, tol=1e-6, halo=None, chunk_len=None, shard=None, posterior_key=None,
                 emission_factory=None, carry_in=None, mstep_fn=None):
        """log_posterior_init: [T,K] array, or None with posterior_key = (key, random_scale, t_offset, T_total):
        the reference's random initial posterior (core.py:571-583) drawn on the device.
        emission_factory / carry_in: see EStep (other observation models, latent-only families);
        mstep_fn(Phi, yw, tw, W) -> tuning [K,N] replaces the Adam M-step (updates W in place; Gaussian families)."""
        self.y = y_dev
        self.Phi = model._dev(tuning_basis)
        W0 = model._dev(model.params)
        if W0.shape != (self.Phi.shape[1], model.n_neuron):
            raise ValueError("params shape %s does not match basis %s" % (tuple(W0.shape), tuple(self.Phi.shape)))
        # weights and Adam moments in one buffer: one copy snapshots / restores the optimiser
        self.state = ops.AdamState.packed(W0)
        self.W = self.state.W
        self._snap = torch.empty_like(self.state.flat)
        self._snap_count = torch.empty_like(self.state.count)
        # One buffer holds everything an EM iteration sums over ranks: the statistics [K, N+1] (column N =
        # sum_t gamma) followed by the E-step's record (log marginal, seam verdict) -> ONE all-reduce per iteration
        K_, N1 = op.K, model.n_neuron + 1
        self.pack = torch.zeros(K_ * N1 + estep.TAIL, dtype=torch.float32, device=self.W.device)
        self.stats = self.pack[:K_ * N1].view(K_, N1)
        self.mstep_fn = mstep_fn
        self.es = EStep(y_dev, op, ma_n, ma_l, likelihood_scale, halo=halo, chunk_len=chunk_len, shard=shard,
                        em_mode=True, tail=self.pack[K_ * N1:], emission_factory=emission_factory, carry_in=carry_in)
        self.shard = self.es.shard
        self.broadcast_mstep = os.environ.get("PMG_MSTEP_BROADCAST", "0") != "0"
        self.prior_std, self.step_size, self.maxiter, self.tol = prior_std, step_size, maxiter, tol
        self._n_mstep = 0
        self._row_len = 2 * int(maxiter) + 4            # loss history | gradient-norm history | final[2] | n_iter | pad
        self._hist = self._new_hist_block()
        self._scratch = torch.zeros((2, self._row_len), dtype=torch.float32, device=self.W.device)
        self._tuning = torch.empty((2, self.Phi.shape[0], model.n_neuron), dtype=torch.float32, device=self.W.device)
        self._tuning_i = 0
        self._spec = None                  # M-step result enqueued ahead for the next iteration (see iteration)
        self.W_iter = self.W
        self._last_repaired = False
        # tensor-core statistics need fp16-exact counts; otherwise the fp32 CUDA-core tiles are used
        self.use_tc = self.es.y16 is not None and self.es.y16.exact
        T_core, K = y_dev.shape[0], op.K
        # fp16 pieces live on the rank's extended block (core + neighbour halos); halo rows stay zero, so
        # the time reduction over the extended block only counts this rank's own bins
        self.gamma16 = ops.new_gamma16(self.es.T, K, y_dev.device) if self.use_tc else None
        self.gamma_lat, self.tw = None, None
        if log_posterior_init is None:
            key, random_scale, t_offset, T_total = posterior_key
            post, _, tw = ops.threefry_posterior_init(T_core, K, key, random_scale, y_dev.device, t_offset, T_total,
                                                      want_post=not self.use_tc, g16=self.gamma16,
                                                      g16_row0=self.es.core.start, want_tw=not self.use_tc)
            self.gamma_lat, self.tw = post, tw
        else:
            gamma_lat = torch.exp(model._dev(log_posterior_init))
            if gamma_lat.shape != (T_core, K):
                raise ValueError("log_posterior_init must be [T, n_latent_bin]")
            if self.use_tc:
                self.gamma16[:, self.es.core] = ops.split_f16(gamma_lat)
            else:
                self.gamma_lat = gamma_lat
                self.tw = gamma_lat.sum(dim=0, dtype=torch.float64).to(torch.float32)

    _HIST_BLOCK = 32

    # ---- M-step plumbing.  The GPU work of "statistics + all-reduce + M-step" (`_mstep_enqueue`) touches only
    # buffers fixed at construction, chosen by the parity of `_tuning_i`: tuning[p], the packed result row
    # scratch[p], the optimiser state in place.  That makes it replayable inside a CUDA graph.  The bookkeeping
    # that differs from iteration to iteration (history row, counters) is `_mstep_commit`, always eager.
    def _new_hist_block(self):
        return torch.empty((self._HIST_BLOCK, self._row_len), dtype=torch.float32, device=self.W.device)

    def _row_views(self, row):
        """(loss_hist[maxiter], err_hist[maxiter], n_iter[1] int32, final[2]) inside one packed fp32 row"""
        mi = int(self.maxiter)
        return row[:mi], row[mi:2 * mi], row[2 * mi + 2:2 * mi + 3].view(torch.int32), row[2 * mi:2 * mi + 2]

    def _mstep_enqueue(self, with_record=False):
        """Sufficient statistics of the current posterior + the Adam M-step (reference core.py:807-810) into the
        buffers of parity 1 - _tuning_i.  No Python state changes.
        with_record: the E-step's record behind the statistics is final and travels in the same all-reduce."""
        p = 1 - self._tuning_i
        N = self.stats.shape[1] - 1
        if self.use_tc:
            # reference core.py:807; the ones column of the fp16 counts makes column N = sum_t gamma
            ops.atb_f16(self.gamma16, self.es.y16, self.es.K, out=self.stats)
        else:
            ops.atb(self.gamma_lat, self.y, out=self.stats[:, :N])
            self.stats[:, N] = self.tw
        # time-sharded ranks: one all-reduce (fp32 on the wire, in place, no packing copies)
        self.shard.allreduce_flat_sum_(self.pack if with_record else self.pack[:self.stats.numel()])
        ops.phase("stats")
        tun = self._tuning[p]
        if self.mstep_fn is not None:
            tun.copy_(self.mstep_fn(self.Phi, self.stats[:, :N], self.stats[:, N], self.W))
        else:
            lh, eh, ni, fin = self._row_views(self._scratch[p])
            ops.mstep_adam(self.Phi, self.stats[:, :N], self.stats[:, N], self.W, self.state, self.prior_std,
                           self.step_size, self.maxiter, self.tol, out=(lh, eh, ni, fin, tun))   # reference core.py:810
        if self.shard.active and self.broadcast_mstep:
            # The M-step is replicated: every rank runs the same deterministic kernel on the bit-identical result
            # of the all-reduce, so tuning and optimiser state agree bit for bit without communication (ranks
            # recompute their neighbours' halo bins and verify boundary seams at 1e-5; a divergence would show up
            # there).  PMG_MSTEP_BROADCAST=1 restores the explicit broadcast of rank 0's result (debugging).
            st = self.state
            parts = [tun, self.W, st.mu, st.nu]
            flat = torch.cat([t.reshape(-1) for t in parts] + [st.count.to(torch.float32)])
            self.shard.broadcast_(flat, 0)
            o = 0
            for t in parts:
                n = t.numel()
                t.copy_(flat[o:o + n].view(t.shape))
                o += n
            st.count.copy_(flat[o:o + 1].to(torch.int32))
        ops.phase("mstep")

    def _mstep_commit(self):
        """Adopts the M-step `_mstep_enqueue` produced: flips the parity, files the result row in the history
        (nothing that outlives an iteration is allocated per iteration: histories live in blocks of _HIST_BLOCK
        rows) and returns (loss_hist, err_hist, n_iter, final, tuning) as device tensors."""
        self._tuning_i ^= 1
        p = self._tuning_i
        tun = self._tuning[p]
        if self.mstep_fn is not None:
            return (None, None, None, None, tun)
        slot = self._n_mstep % self._HIST_BLOCK
        if slot == 0 and self._n_mstep > 0:
            self._hist = self._new_hist_block()
        self._n_mstep += 1
        row = self._hist[slot]
        row.copy_(self._scratch[p])
        return self._row_views(row) + (tun,)

    def _snapshot(self):
        self._snap.copy_(self.state.flat)
        self._snap_count.copy_(self.state.count)

    def _rollback(self):
        self.state.flat.copy_(self._snap)
        self.state.count.copy_(self._snap_count)

    def _spec_enqueue(self):
        """GPU work enqueued behind an E-step's backward pass, before its verdict is known: snapshot of the
        optimiser state, then the next iteration's statistics + M-step (with the E-step's record in the all-reduce)."""
        self._snapshot()
        self._mstep_enqueue(with_record=True)

    def iteration(self, want_gamma=False, want_dyn=False, want_gamma_lat=False, speculate=False):
        """want_gamma_lat: also return the fp32 latent posterior (always produced on the fp32 path).
        The returned tuning (m_res[4]) is one of two buffers; the iteration after the next overwrites it.

        speculate=True: the statistics GEMM and the M-step of the NEXT iteration are enqueued right behind this
        iteration's backward pass, before the launching thread waits for the seam verdict, so the GPU has work
        while the host synchronises (the one synchronisation per EM iteration).  They only read what the
        backward pass wrote; if a seam then fails and chains are re-run by the host, the optimiser state is restored
        from a snapshot and the next iteration recomputes them.  Pass False for the last iteration of a fit.
        In that steady state everything from the emission GEMM to the M-step is a fixed launch sequence on fixed
        buffers: the E-step captures it into a CUDA graph (one per buffer parity and warm-up plan) and replays it."""
        # (not right after an iteration that needed host repairs: the next one probably does too, and a rolled
        # back M-step is wasted work)
        spec_ok = bool(speculate and self.use_tc and not self._last_repaired and self.mstep_fn is None
                       and os.environ.get("PMG_NO_SPECULATE", "0") == "0")
        if self._spec is not None:
            m_res, self._spec = self._spec, None
        else:
            self._mstep_enqueue()
            m_res = self._mstep_commit()
        res = self.es.run(m_res[4], want_gamma=want_gamma, want_gamma_lat=(want_gamma_lat or not self.use_tc),
                          want_dyn=want_dyn, want_r=False, gamma16=self.gamma16,
                          before_sync=self._spec_enqueue if spec_ok else None, graph_ok=spec_ok)
        self._last_repaired = bool(res.repaired)
        # GLM weights that produced THIS iteration's tuning (self.W may already hold the next M-step's result)
        self.W_iter = self._snap[0] if spec_ok else self.W
        if spec_ok:
            if res.repaired:
                self._rollback()
            else:
                self._spec = self._mstep_commit()
        self.gamma_lat = res.gamma_lat                             # reference core.py:668
        if res.tw is not None:
            self.tw = res.tw
        return res, m_res                                          # res.log_marginal is global already


class PoissonGPLVMJump1D:
    """Poisson GPLVM with a smooth 1-D latent plus jumps (reference core.py:746)."""

    def __init__(self, n_neuron, n_latent_bin=100, tuning_lengthscale=1., param_prior_std=1.,
                 movement_variance=1.,
                 explained_variance_threshold_basis=0.999,
                 rng_init_int=123,
                 w_init_variance=1.,
                 w_init_mean=0.,
                 p_move_to_jump=0.01,
                 p_jump_to_move=0.01,
                 basis_type='rbf',
                 custom_tuning_kernel=None,
                 custom_transition_kernel=None,
                 smoothness_penalty=0.,
                 device=None):
        if basis_type not in ('rbf', 'custom_kernel'):
            raise ValueError("basis_type %r is not supported (the reference disables bspline too, core.py:57-59)"
                             % (basis_type,))
        self.n_latent_bin = n_latent_bin
        self.tuning_lengthscale = tuning_lengthscale
        self.param_prior_std = param_prior_std
        self.movement_variance = movement_variance
        self.p_move_to_jump = p_move_to_jump
        self.p_jump_to_move = p_jump_to_move
        self.explained_variance_threshold_basis = explained_variance_threshold_basis
        self.rng_init_int = rng_init_int
        self.rng_init = jaxprng.PRNGKey(rng_init_int)
        self.n_neuron = n_neuron
        self.possible_latent_bin = np.arange(n_latent_bin)
        self.possible_dynamics = np.arange(2)
        self.w_init_variance = w_init_variance
        self.w_init_mean = w_init_mean
        self.custom_transition_kernel = custom_transition_kernel
        self.basis_type = basis_type
        self.tuning_basis = gpk.generate_basis(tuning_lengthscale, n_latent_bin, explained_variance_threshold_basis,
                                               include_bias=True, basis_type=basis_type,
                                               custom_kernel=custom_tuning_kernel)
        self.n_basis = self.tuning_basis.shape[1]
        self.smoothness_penalty = smoothness_penalty
        self.ma_neuron_default = np.ones(n_neuron, dtype=np.float32)
        self.ma_latent_default = np.ones(n_latent_bin, dtype=np.float32)
        self._device = device
        self.adam_runner = None
        self.opt_state_init_fun = None
        self.initialize_params(self.rng_init)

    # ------------------------------------------------------------------ plumbing
    @property
    def device(self):
        if self._device is None:
            if not torch.cuda.is_available():
                raise RuntimeError("poor_man_gplvm_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
            self._device = torch.device("cuda", torch.cuda.current_device())
        return torch.device(self._device)

    def __getstate__(self):
        state = self.__dict__.copy()
        state['adam_runner'] = None
        state['opt_state_init_fun'] = None
        state.pop('_opt_state', None)          # device tensors; fit_em re-initialises Adam anyway (core.py:847)
        state.pop('_pack_cache', None)         # device tensors; rebuilt on demand
        return state

    def __setstate__(self, state):
        self.__dict__.update(state)

    def _dev(self, a, dtype=torch.float32):
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous()
        if isinstance(a, hostio.LazyHostArray):
            return a.device_tensor().to(device=self.device, dtype=dtype).contiguous()
        return hostio.to_device(np.asarray(a), self.device).to(dtype).contiguous()

    @staticmethod
    def _host(t, out=None):
        """device tensor -> NumPy (pinned, pipelined copy for the T-sized arrays)"""
        return hostio.to_numpy(t, out=out) if isinstance(t, torch.Tensor) else np.asarray(t)

    # ------------------------------------------------------------------ hooks of the other families (families.py)
    def _emission_factory(self, hyperparam):
        """callable(y_ext, ma_neuron) -> emission operand, or None for the Poisson model of this class"""
        return None

    def _mstep_fn(self, hyperparam):
        """callable(Phi, yw, tw, W) -> tuning replacing the Adam M-step, or None"""
        return None

    # ------------------------------------------------------------------ reference API
    @_on_device
    def get_tuning(self, params, hyperparam, tuning_basis):
        """softplus(basis @ params)  (reference core.py:772-774).  NumPy in -> NumPy out."""
        Phi, W = self._dev(tuning_basis), self._dev(params)
        return self._host(ops.tuning_softplus(Phi, W))

    def initialize_params(self, key):
        """reference core.py:429-437: normal(key, (n_basis, n_neuron)) * sqrt(w_init_variance) + w_init_mean with
        jax.random's bit stream (jaxprng.py).  (The tuning basis comes from an SVD whose sign convention is
        backend dependent in the reference as well; inject ``tuning_basis`` for run-for-run reproduction.)"""
        params = (jaxprng.normal(key, (self.n_basis, self.n_neuron)) * np.float32(np.sqrt(self.w_init_variance))
                  + np.float32(self.w_init_mean)).astype(np.float32)
        self.params = params
        # softplus(Phi W) on the host: the constructor must work without touching the GPU
        self.tuning = np.logaddexp(self.tuning_basis @ params, np.float32(0)).astype(np.float32)
        return self.params, self.tuning

    @_on_device
    def init_latent_posterior(self, T, key, random_scale=0.1):
        """reference core.py:571-583 with jax.random's bit stream: uniform(key, (T, K)) * random_scale, row
        normalised.  Returns (log_posterior, posterior) as NumPy arrays; large draws run on the device."""
        K = self.n_latent_bin
        if T * K > _HOST_PRNG_MAX and torch.cuda.is_available():
            post, logp, _ = ops.threefry_posterior_init(T, K, key, random_scale, self.device, want_post=True,
                                                        want_log=True)
            return self._host(logp), self._host(post)
        posterior = jaxprng.uniform(key, (T, K)) * np.float32(random_scale)
        posterior = posterior / posterior.sum(axis=1, keepdims=True)
        with np.errstate(divide="ignore"):
            log_posterior = np.log(posterior)            # log(0) = -inf, the reference's -1e40 in fp32
        return log_posterior, posterior

    def _transition_pack(self, hyperparam):
        mv = hyperparam.get('movement_variance', self.movement_variance)
        pmj = hyperparam.get('p_move_to_jump', self.p_move_to_jump)
        pjm = hyperparam.get('p_jump_to_move', self.p_jump_to_move)
        # K x K host work (kernel matrices, band factorisation, stationary solve): a few ms, reused by repeated
        # fit / decode calls with the same dynamics
        ck = self.custom_transition_kernel
        ck_key = None if ck is None else hash(np.ascontiguousarray(np.asarray(ck, dtype=np.float32)).tobytes())
        key = (float(mv), float(pmj), float(pjm), ck_key, self.n_latent_bin, str(self.device))
        cached = getattr(self, "_pack_cache", None)
        if cached is not None and cached[0] == key:
            return cached[1]
        P, logP, M, logM = gpk.create_transition_prob_1d(self.possible_latent_bin, self.possible_dynamics, mv, pmj, pjm,
                                                         custom_kernel=self.custom_transition_kernel)
        host = gpk.move_operator_host(self.n_latent_bin, mv, self.custom_transition_kernel, p_move_to_jump=pmj)
        op = ops.MoveOperator(host, M, self.device, P0=P[0])
        self._pack_cache = (key, (P, logP, M, logM, op))
        return P, logP, M, logM, op

    def _masks(self, ma_neuron, ma_latent, T):
        if ma_neuron is None:
            ma_neuron = self.ma_neuron_default
        if ma_latent is None:
            ma_latent = self.ma_latent_default
        ma_n = self._dev(ma_neuron)
        if ma_n.dim() == 2 and tuple(ma_n.shape) != (T, self.n_neuron):
            raise ValueError("ma_neuron must be [n_neuron] or [T, n_neuron], got %s" % (tuple(ma_n.shape),))
        if ma_n.dim() == 1 and ma_n.shape[0] != self.n_neuron:
            raise ValueError("ma_neuron must be [n_neuron] or [T, n_neuron], got %s" % (tuple(ma_n.shape),))
        return ma_n, self._dev(ma_latent)

    def _transition_counts(self, es, res, logP, logM):
        """log sum_t xi_t (reference decoder.py:215-221) = log(M * P * (alpha^T r)): one time-reduction GEMM
        over this rank's (t, t+1) pairs, summed over ranks, then the [2,2,K,K] epilogue."""
        K = self.n_latent_bin
        c = res.core
        hi = c.stop - 1 if es.shard.is_last else c.stop          # pairs (t, t+1) with t in [c.start, hi)
        if hi > c.start and res.xi16 is not None:
            # the backward pass wrote both operands as bf16 hi/lo pieces: tensor cores, three products
            G = ops.atb_bf16x2_pieces(res.xi16, c.start, hi - c.start)
        elif hi > c.start:
            A = res.alpha_ext.view(-1, 2 * K)[c.start:hi]
            R = res.r_ext.view(-1, 2 * K)[c.start + 1:hi + 1]
            # long recordings: tensor cores on bf16 hi/lo pieces (three products); short ones: fp32 CUDA cores
            G = ops.atb_bf16x2(A, R) if hi - c.start >= ops.XI_TC_MIN_BINS else ops.atb(A, R)
        else:
            G = torch.zeros((2 * K, 2 * K), dtype=torch.float32, device=self.device)
        es.shard.allreduce_sum_(G)
        return ops.xi_finalize(G, self._dev(logP), logM)

    @_on_device
    def _decode_latent(self, y, tuning, hyperparam, log_latent_transition_kernel_l=None,
                       log_dynamics_transition_kernel=None, ma_neuron=None, ma_latent=None, likelihood_scale=1.,
                       n_time_per_chunk=10000, return_device=False, _want_r=True):
        """reference core.py:777-786: returns the 6-tuple (log_acausal_posterior_all [T,2,K],
        log_marginal_final, log_causal_posterior_all [T,2,K], log_one_step_predictive_marginals [T],
        log_accumulated_joint_total [2,2,K,K], log_likelihood_all [T,K]).  The transition kernels are
        rebuilt from ``hyperparam``/attributes (the log arguments are accepted for signature
        compatibility); ``n_time_per_chunk`` is a numerical no-op in the reference and ignored here."""
        y, _ = _unwrap_tsd(y)
        y_dev = self._dev(y)
        P, logP, M, logM, op = self._transition_pack(hyperparam)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, y_dev.shape[0])
        es = EStep(y_dev, op, ma_n, ma_l, likelihood_scale, emission_factory=self._emission_factory(hyperparam))
        res = es.run(self._dev(tuning), want_gamma=True, want_gamma_lat=False, want_dyn=False, want_r=_want_r,
                     xi16_ok=y_dev.shape[0] - 1 >= ops.XI_TC_MIN_BINS)
        log_acc = None
        if _want_r and y_dev.shape[0] > 1:
            log_acc = self._transition_counts(es, res, logP, logM)
        out = (torch.log(res.gamma), res.log_marginal.to(torch.float32), torch.log(res.alpha), res.lmr, log_acc,
               res.ll)
        if return_device:
            return out
        return tuple(None if o is None else self._host(o) for o in out)

    @_on_device
    def decode_latent(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None, likelihood_scale=1.,
                      n_time_per_chunk=10000, t_l=None, return_device=False, time_sharded=False, group=None):
        """reference core.py:454-497 (same keys).  time_sharded=True (under torch.distributed): ``y`` is this
        rank's contiguous block of time bins; T-sized results cover that block, scalars and the transition
        statistics are global."""
        y, t_in = _unwrap_tsd(y)
        if t_in is not None:
            t_l = t_in
        if tuning is None:
            tuning = self.tuning
        y_dev = self._dev(y)
        T, K = y_dev.shape[0], self.n_latent_bin
        P, logP, M, logM, op = self._transition_pack(hyperparam)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, T)
        es = EStep(y_dev, op, ma_n, ma_l, likelihood_scale, shard=TimeShard(group) if time_sharded else None,
                   emission_factory=self._emission_factory(hyperparam))
        res = es.run(self._dev(tuning), want_gamma=True, want_gamma_lat=True, want_dyn=True,
                     want_r=(T > 1 or es.shard.active), xi16_ok=T - 1 >= ops.XI_TC_MIN_BINS)
        conv = (lambda t: t) if return_device else self._host
        # the reference leaves these on the device as jax arrays (core.py:489, decoder.py:360-375)
        lazy = (lambda t: t) if return_device else hostio.LazyHostArray
        decoding_res = {'log_posterior_all': conv(torch.log(res.gamma)),
                        'log_marginal_final': float(res.log_marginal.item()),
                        'posterior_all': conv(res.gamma),
                        'posterior_latent_marg': _rewrap_tsd(conv(res.gamma_lat), t_l),
                        'posterior_dynamics_marg': _rewrap_tsd(conv(res.dyn_marg), t_l),
                        'log_one_step_predictive_marginals_all': lazy(res.lmr),
                        'log_likelihood_all': conv(res.ll)}
        if T > 1 or es.shard.active:
            log_acc = self._transition_counts(es, res, logP, logM)
            tp = compute_transition_posterior_prob(log_acc)
            decoding_res.update({k: lazy(v) for k, v in tp.items()})
        self._last_estep_info = {"n_chain": res.plan.n_chain, "relay_fwd": res.n_relay_fwd,
                                 "relay_bwd": res.n_relay_bwd, "seam_err_fwd": res.seam_err_fwd,
                                 "seam_err_bwd": res.seam_err_bwd}
        return decoding_res

    def _viterbi_inputs(self, y, ma_neuron, ma_latent):
        """Shape checks of decode_latent_viterbi, on the host before any device work."""
        shp = tuple(getattr(y, "shape", np.shape(y)))
        if len(shp) != 2 or shp[0] < 1 or shp[1] != self.n_neuron:
            raise ValueError("y must be [T, n_neuron=%d] with T >= 1, got shape %s" % (self.n_neuron, shp))
        if ma_neuron is not None:
            ms = tuple(getattr(ma_neuron, "shape", np.shape(ma_neuron)))
            if ms not in ((self.n_neuron,), (shp[0], self.n_neuron)):
                raise ValueError("ma_neuron must be [n_neuron] or [T, n_neuron], got %s" % (ms,))
        if ma_latent is not None:
            m = ma_latent.detach().cpu().numpy() if isinstance(ma_latent, torch.Tensor) else np.asarray(ma_latent)
            if m.shape != (self.n_latent_bin,):
                raise ValueError("ma_latent must be [n_latent_bin=%d], got %s" % (self.n_latent_bin, m.shape))
            if not np.any(m != 0):
                raise ValueError("ma_latent masks every latent bin: no path has nonzero probability")

    def _viterbi(self, y, tuning, hyperparam, ma_neuron, ma_latent, likelihood_scale, carry_in_of,
                 time_sharded=False, group=None):
        """(flat path [T] int64 on the device, log_joint_map float); carry_in_of(op): the message in front of bin 0
        (time-sharded: in front of rank 0's block; the other ranks' chain 0 starts from the left neighbour)."""
        self._viterbi_inputs(y, ma_neuron, ma_latent)
        if tuning is None:
            tuning = self.tuning
        y_dev = self._dev(y)
        P, logP, M, logM, op = self._transition_pack(hyperparam)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, y_dev.shape[0])
        es = EStep(y_dev, op, ma_n, ma_l, likelihood_scale, emission_factory=self._emission_factory(hyperparam),
                   carry_in=carry_in_of(op), shard=TimeShard(group) if time_sharded else None)
        res = viterbi.run(es, self._dev(tuning))
        self._last_estep_info = {"n_chain": res.n_chain, "fix_fwd": res.n_fix, "relay_fwd": res.n_relay,
                                 "relay_fwd_boundary": res.n_relay_boundary, "seam_err_fwd": res.seam_err}
        return res.path.to(torch.int64), float(res.log_joint_map.item())

    @_on_device
    def decode_latent_viterbi(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None,
                              likelihood_scale=1., n_time_per_chunk=10000, t_l=None, return_device=False,
                              time_sharded=False, group=None):
        """Most probable joint (dynamics, latent) path: argmax over paths of p(path, y).  Beyond the reference.

        Joint state s = (d, x), d in {0 move, 1 jump}, x in [0, K); transition M[d,d'] P_{d'}[x,x'] with P_0 the move
        kernel of the model (RBF Toeplitz or custom band, as in decode_latent) and P_1 = 1/K.  Bin 0's prior is the
        filter's prior from its carry, so sum over paths of p(path, y) = exp(log_marginal_final) of decode_latent: the
        start is marginalised, not maximised.  Emission: likelihood_scale * log-likelihood, as in the filter;
        ma_latent == 0 bins have likelihood 0 and never lie on the path.  Exact ties resolve to the smallest flat
        index d*K + x, in every predecessor max and in the final argmax.

        Returns ``map_latent`` and ``map_dynamics`` (int64 [T]; a Tsd when y is a TsdFrame or t_l is given) and
        ``log_joint_map`` = log p(path*, y).  ``n_time_per_chunk`` is accepted for signature symmetry with
        decode_latent and ignored (the time-parallel chunking is chosen by the E-step plan; the path does not depend
        on it beyond the seam tolerance).  ma_neuron: [N] or [T, N].  An ma_latent without a nonzero entry raises
        ValueError.

        time_sharded=True (under torch.distributed, every rank of ``group`` calls together): ``y`` (and a [T, N]
        ma_neuron) is this rank's contiguous block of bins; ``map_latent`` / ``map_dynamics`` cover that block and
        ``log_joint_map`` is the global value, identical on every rank.  The path is the single-device path."""
        y, t_in = _unwrap_tsd(y)
        if t_in is not None:
            t_l = t_in
        path, lj = self._viterbi(y, tuning, hyperparam, ma_neuron, ma_latent, likelihood_scale, lambda op: None,
                                 time_sharded, group)
        K = self.n_latent_bin
        conv = (lambda t: t) if return_device else self._host
        return {'map_latent': _rewrap_tsd_1d(conv(path % K), t_l),
                'map_dynamics': _rewrap_tsd_1d(conv(path // K), t_l),
                'log_joint_map': lj}

    @_on_device
    def decode_latent_naive_bayes(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None,
                                  likelihood_scale=1., n_time_per_chunk=10000, dt_l=1., t_l=None,
                                  return_device=False):
        """reference core.py:788-792 -> :499-524 (``likelihood_scale`` accepted and ignored, as there)."""
        y, t_in = _unwrap_tsd(y)
        if t_in is not None:
            t_l = t_in
        if tuning is None:
            tuning = self.tuning
        y_dev = self._dev(y)
        T = y_dev.shape[0]
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, T)
        # dt_l: scalar or per-bin [T] (reference decoder.py:124 broadcasts it to [T])
        dt_dev = self._dev(dt_l).reshape(-1)
        if dt_dev.numel() not in (1, T):
            raise ValueError("dt_l must be a scalar or have one entry per time bin")
        if not bool((dt_dev > 0).all()):
            # the reference keeps log(tuning*dt + 1e-20) finite at dt = 0; the GEMM form separates log(dt)
            raise ValueError("dt_l must be positive (a bin of zero or negative duration has no likelihood)")
        factory = self._emission_factory(hyperparam)
        if dt_dev.numel() == T and T > 1 and bool((dt_dev != dt_dev[0]).any()):
            if factory is not None:
                raise ValueError("per-bin dt_l is implemented for the Poisson model only")
            em = ops.EmissionOperands(y_dev, ma_n, dt_l=dt_dev)
            dt = 1.0
        else:
            em = factory(y_dev, ma_n) if factory is not None else ops.EmissionOperands(y_dev, ma_n)
            dt = float(dt_dev[0].item()) if dt_dev.numel() else 1.0
        ll = em.loglik(self._dev(tuning), ma_l, dt)
        log_post, lml, post = ops.naive_bayes_normalize(ll, want_post=True)
        conv = (lambda t: t) if return_device else self._host
        return {'log_posterior_latent': conv(log_post),
                'log_marginal_l': conv(lml),
                'log_marginal_total': float(lml.sum(dtype=torch.float64).item()),
                'posterior_latent': _rewrap_tsd(conv(post), t_l),
                'll_per_pos_l': conv(ll)}

    @_on_device
    def m_step(self, param_curr, y, log_posterior_curr, tuning_basis, hyperparam, opt_state_curr=None,
               m_step_step_size=0.01, m_step_maxiter=1000, m_step_tol=1e-6):
        """reference core.py:802-827: sufficient statistics + Adam loop.  NumPy/torch in, dict out."""
        y_dev = self._dev(_unwrap_tsd(y)[0])
        post = torch.exp(self._dev(log_posterior_curr))
        yw = ops.atb(post, y_dev)
        tw = post.sum(dim=0, dtype=torch.float64).to(torch.float32)
        W = self._dev(param_curr).clone()
        state = opt_state_curr if isinstance(opt_state_curr, ops.AdamState) else ops.AdamState(W)
        prior_std = hyperparam.get('param_prior_std', self.param_prior_std)
        lh, eh, n_it, fin, tuning = ops.mstep_adam(self._dev(tuning_basis), yw, tw, W, state, prior_std,
                                                   m_step_step_size, m_step_maxiter, m_step_tol)
        n = int(n_it.item())
        return {'params': self._host(W), 'opt_state': state, 'n_iter': n,
                'final_loss': float(fin[0].item()), 'final_error': float(fin[1].item()),
                'loss_history': self._host(lh[:n]), 'error_history': self._host(eh[:n])}

    @_on_device
    def fit_em(self, y, hyperparam={}, key=0,
               n_iter=20, log_posterior_init=None, ma_neuron=None, ma_latent=None,
               n_time_per_chunk=10000, dt=1., likelihood_scale=1.,
               save_every=None,
               m_step_step_size=0.01, m_step_maxiter=1000, m_step_tol=1e-6,
               posterior_init_kwargs={'random_scale': 0.1}, verboase=True, return_device=False,
               time_sharded=False, group=None,
               **kwargs):
        """reference core.py:829-849 -> :592-713.  Per iteration: M-step (statistics + Adam) on the
        current posterior, tuning, E-step; ``em_res`` has the reference's keys.
        time_sharded=True (one process per GPU under torch.distributed): ``y`` and ``log_posterior_init`` are
        this rank's contiguous block of time bins; T-sized results cover that block, while ``params``,
        ``tuning`` and the log marginals are global and identical on every rank."""
        y_in, t_l = _unwrap_tsd(y)
        hyperparam_ = dict(hyperparam)
        prior_std = hyperparam_.get('param_prior_std', self.param_prior_std)
        hyperparam_['param_prior_std'] = prior_std
        hyperparam_['smoothness_penalty'] = hyperparam_.get('smoothness_penalty', self.smoothness_penalty)

        self.tuning_lengthscale = hyperparam_.get('tuning_lengthscale', self.tuning_lengthscale)
        self.movement_variance = hyperparam_.get('movement_variance', self.movement_variance)
        self.p_move_to_jump = hyperparam_.get('p_move_to_jump', self.p_move_to_jump)
        self.p_jump_to_move = hyperparam_.get('p_jump_to_move', self.p_jump_to_move)

        tm = _Timing()
        T, K = int(np.shape(y_in)[0]), self.n_latent_bin
        y_dev = self._dev(y_in)                       # the one host->device copy of the spikes
        tm.mark("h2d_y")
        if save_every is None:
            save_every = n_iter
        P, logP, M, logM, op = self._transition_pack(hyperparam_)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, T)
        if 'tuning_lengthscale' in hyperparam:
            tuning_basis = gpk.generate_basis(self.tuning_lengthscale, K, self.explained_variance_threshold_basis,
                                              include_bias=True)
        else:
            tuning_basis = self.tuning_basis
        shard = TimeShard(group) if time_sharded else None
        posterior_key = None
        if log_posterior_init is None:
            # the reference draws uniform(key, (T, K)) on its device (core.py:579); here the same bit stream is
            # generated on the GPU straight into the operands of the first M-step; em_res['log_posterior_init']
            # regenerates it on demand.  A time-sharded rank draws its rows of the global [T_total, K] array.
            random_scale = posterior_init_kwargs.get('random_scale', 0.1)
            t_offset, T_total = (shard.block_offset(T) if shard is not None else (0, T))
            posterior_key = (jaxprng.as_key(key), random_scale, t_offset, T_total)
            dev_ = self.device
            log_posterior_init = hostio.LazyHostArray(
                None, shape=(T, K), device=dev_, producer=lambda: ops.threefry_posterior_init(
                    T, K, posterior_key[0], random_scale, dev_, t_offset, T_total, want_log=True)[1])
            loop_init = None
        else:
            loop_init = log_posterior_init
        mstep_fn = self._mstep_fn(hyperparam_)
        loop = EMLoop(self, y_dev, op, ma_n, ma_l, likelihood_scale, tuning_basis, loop_init, prior_std,
                      m_step_step_size, m_step_maxiter, m_step_tol, shard=shard, posterior_key=posterior_key,
                      emission_factory=self._emission_factory(hyperparam_), mstep_fn=mstep_fn)
        self.opt_state_init_fun = ops.AdamState
        W, state, es = loop.W, loop.state, loop.es
        tm.mark("setup")
        # the host copies of the T-sized results are allocated now and their pages faulted in by background
        # threads while the EM iterations run on the GPU (after the setup above: the populate calls hold the
        # process's memory-map lock, which stalls every allocation the setup makes on the main thread)
        bufs = None
        if not return_device and n_iter > 0 and T * K >= (1 << 22):
            bufs = hostio.HostBuffers([("posterior", (T, 2, K), np.float32), ("latent", (T, K), np.float32),
                                       ("dynamics", (T, 2), np.float32)])

        lml_dev, m_hist = [], []
        saved = {'log_posterior_all_saved': [], 'params_saved': [], 'tuning_saved': [], 'iter_saved': [],
                 'log_marginal_saved': []}
        estep_info = []
        conv = (lambda t: t) if return_device else self._host
        # jax device arrays in the reference (core.py:672-675, :703): copied to the host on first use
        lazy_log = (lambda t: torch.log(t)) if return_device else (lambda t: hostio.LazyHostArray(t, torch.log))
        res = None
        tm.t_it = time.perf_counter()
        for i in range(n_iter):
            tm.iteration()
            last = i == n_iter - 1
            snap = (i % save_every == 0)
            res, m_res = loop.iteration(want_gamma=(last or snap), want_dyn=last, want_gamma_lat=last,
                                        speculate=not last)
            m_hist.append(m_res)
            tuning = m_res[4]
            lml_dev.append(res.log_marginal)
            estep_info.append((res.n_relay_fwd, res.n_relay_bwd, res.seam_err_fwd, res.seam_err_bwd))
            if snap:
                saved['log_posterior_all_saved'].append(lazy_log(res.gamma))
                saved['params_saved'].append(conv(loop.W_iter.clone()))
                saved['tuning_saved'].append(conv(tuning.clone() if return_device else tuning))
                saved['log_marginal_saved'].append(res.log_marginal)
                saved['iter_saved'].append(i)

        tm.iteration()
        tm.mark("em_loop")
        lml_host = torch.stack(lml_dev).cpu().numpy().astype(np.float32) if lml_dev else np.zeros(0, np.float32)
        saved['log_marginal_saved'] = [np.float32(v.item()) for v in saved['log_marginal_saved']]
        if mstep_fn is not None:
            m_hist = []                            # analytic M-step: no optimiser histories (reference core.py:885-892)
        n_its = torch.cat([h[2] for h in m_hist]).cpu().numpy() if m_hist else np.zeros(0, np.int32)
        m_step_res_l = {'n_iter': [int(n) for n in n_its],
                        'final_loss': [float(h[3][0].item()) for h in m_hist],
                        'final_error': [float(h[3][1].item()) for h in m_hist],
                        'loss_history': [self._host(h[0][:int(n)]) for h, n in zip(m_hist, n_its)],
                        'error_history': [self._host(h[1][:int(n)]) for h, n in zip(m_hist, n_its)]}

        self.params = self._host(W)
        self.tuning = self._host(tuning) if n_iter > 0 else self.tuning
        self.log_marginal_final = lml_host[-1] if n_iter > 0 else None
        self.log_latent_transition_kernel_l = logP
        self.log_dynamics_transition_kernel = logM
        self.tuning_basis = tuning_basis
        self._last_estep_info = {"n_chain": es.plan.n_chain, "chunk_len": es.chunk_len, "halo": es.halo,
                                 "per_iter": estep_info, "tensor_core_statistics": bool(loop.use_tc),
                                 "compact_scan": bool(es.compact_ok and loop.use_tc)}
        self._opt_state = state

        em_res = dict(saved)
        em_res.update({'log_posterior_init': log_posterior_init,
                       'params': self.params,
                       'tuning': self.tuning,
                       'log_marginal_l': [v for v in lml_host],
                       'm_step_res_l': m_step_res_l})
        if n_iter > 0:
            take = (lambda n: bufs.take(n)) if bufs is not None else (lambda n: None)
            conv_to = (lambda t, n: t) if return_device else (lambda t, n: self._host(t, out=take(n)))
            em_res.update({'log_posterior_final': lazy_log(res.gamma),
                           'log_marginal': lml_host[-1],
                           'posterior': conv_to(res.gamma, "posterior"),
                           'posterior_latent_marg': _rewrap_tsd(conv_to(res.gamma_lat, "latent"), t_l),
                           'posterior_dynamics_marg': _rewrap_tsd(conv_to(res.dyn_marg, "dynamics"), t_l)})
        if bufs is not None:
            bufs.close()
        tm.mark("outputs")
        tm.report()
        return em_res

    def predict_expected_rate(self, post_latent_marg, tuning=None):
        """reference core.py:716-733: rate[t,n] = sum_p post[t,p] tuning[p,n]."""
        if tuning is None:
            tuning = self.tuning
        vals, t_l = _unwrap_tsd(post_latent_marg)
        rate = np.asarray(self._host(vals)) @ np.asarray(self._host(tuning))
        return _rewrap_tsd(rate, t_l)

    def sample_latent(self, T, key=0, movement_variance=1, p_move_to_jump=0.01, p_jump_to_move=0.01,
                      init_dynamics=None, init_latent=None):
        """reference core.py:526-555 (NumPy PRNG stream).  Returns [T,2] = (dynamics, latent)."""
        rng = np.random.default_rng(_seed_from_key(key))
        P, _, M, _ = gpk.create_transition_prob_1d(self.possible_latent_bin, self.possible_dynamics,
                                                   movement_variance, p_move_to_jump, p_jump_to_move)
        P = P.astype(np.float64); M = M.astype(np.float64)
        P /= P.sum(axis=2, keepdims=True); M /= M.sum(axis=1, keepdims=True)
        d = int(rng.integers(0, 2)) if init_dynamics is None else int(init_dynamics)
        x = int(rng.integers(0, self.n_latent_bin)) if init_latent is None else int(init_latent)
        out = np.empty((T, 2), dtype=np.int64)
        for t in range(T):
            d = int(rng.choice(2, p=M[d]))
            x = int(rng.choice(self.n_latent_bin, p=P[d][x]))
            out[t] = (d, x)
        return out

    def sample_y(self, latent_l, hyperparam={}, tuning=None, dt=1., key=10):
        """reference core.py:794-800."""
        if tuning is None:
            tuning = self.tuning
        rng = np.random.default_rng(_seed_from_key(key))
        return rng.poisson(np.asarray(self._host(tuning))[np.asarray(latent_l)] * dt)

    def sample(self, T, hyperparam={}, key=0, init_dynamics=None, init_latent=None, dt=1., tuning=None):
        """reference core.py:558-569."""
        mv = hyperparam.get('movement_variance', self.movement_variance)
        pmj = hyperparam.get('p_move_to_jump', self.p_move_to_jump)
        pjm = hyperparam.get('p_jump_to_move', self.p_jump_to_move)
        seed = _seed_from_key(key)
        latent_l = self.sample_latent(T, seed, mv, pmj, pjm, init_dynamics, init_latent)
        y_l = self.sample_y(latent_l[:, 1], hyperparam, tuning, dt, seed + 1)
        return latent_l, y_l
