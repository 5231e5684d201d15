"""The reference's other model families on the same kernels (SURVEY.md section 8(f) row F2).

* ``GaussianGPLVMJump1D`` (reference core.py:852-916): the jump model with a Gaussian observation model
  (decoder.py:50-57), linear tuning (fit_tuning_helper.py:11-17) and the analytic ridge M-step
  (fit_tuning_helper.py:44-61).
* ``PoissonGPLVM1D`` / ``GaussianGPLVM1D`` (reference core.py:919-1093 on ``AbstractGPLVM1D`` :76-373 and
  ``decoder_latentonly.py``): latent only, no dynamics dimension.  They run on the jump kernels with a degenerate
  dynamics chain -- M = identity and all mass on the "move" state -- which reproduces the D = 1 recursion exactly
  (the jump state carries probability zero for ever); results are returned without the dynamics axis.

Observations of the Gaussian models are real-valued: emission through ``pmg_emission_gaussian`` (fp32 CUDA cores),
statistics and scans through the fp32 kernels (the fp16/tcgen05 path needs exact integer counts).

Limitation of the latent-only models (linear-space filter in fp32): the reference's log-space filter stays finite
when an observation lies where the smooth prior has underflowed (a latent that moved many bins in one step); here
the one-step normaliser is then zero and ``RuntimeError`` is raised -- such data calls for the jump models.
"""
from __future__ import annotations

import numpy as np
import torch

from . import gp_kernel as gpk
from . import hostio
from . import jaxprng
from . import ops
from . import viterbi
from .core import (EMLoop, PoissonGPLVMJump1D, _on_device, _rewrap_tsd, _rewrap_tsd_1d, _seed_from_key,
                   _unwrap_tsd)
from .estep import EStep


def _gaussian_mstep(noise_std, prior_std):
    """reference fit_tuning_helper.py:44-61: W = (Phi^T diag(tw) Phi / s^2 + I / prior^2)^-1 Phi^T yw / s^2.
    A B x B solve (B <= K): torch.linalg on the device, once per EM iteration."""
    def fn(Phi, yw, tw, W):
        nv = float(noise_std) ** 2
        P64 = Phi.double()
        H = (P64.T * tw.double().unsqueeze(0)) @ P64 / nv
        H = H + torch.eye(P64.shape[1], dtype=torch.float64, device=Phi.device) / float(prior_std) ** 2
        rhs = P64.T @ yw.double() / nv
        W.copy_(torch.linalg.solve(H, rhs).to(torch.float32))
        return Phi @ W                                   # linear tuning, fit_tuning_helper.py:11-17
    return fn


class _GaussianMixin:
    """Gaussian observation model: emission operand, analytic M-step, linear tuning."""
    noise_std = 0.5

    def _noise(self, hyperparam):
        return float(hyperparam.get('noise_std', self.noise_std))

    def _emission_factory(self, hyperparam):
        s = self._noise(hyperparam)
        return lambda y_ext, ma_neuron: ops.GaussianEmission(y_ext, ma_neuron, noise_std=s)

    def _mstep_fn(self, hyperparam):
        return _gaussian_mstep(self._noise(hyperparam), hyperparam.get('param_prior_std', self.param_prior_std))

    @_on_device
    def get_tuning(self, params, hyperparam, tuning_basis):
        """basis @ params (reference fit_tuning_helper.py:11-17)."""
        return (np.asarray(tuning_basis, np.float32) @ np.asarray(params, np.float32)).astype(np.float32)

    def _init_tuning(self, params):
        return (self.tuning_basis @ params).astype(np.float32)

    def sample_y(self, latent_l, hyperparam={}, tuning=None, dt=1., key=10):
        """reference core.py:885-893 (NumPy stream)."""
        if tuning is None:
            tuning = self.tuning
        rng = np.random.default_rng(_seed_from_key(key))
        rate = np.asarray(self._host(tuning))[np.asarray(latent_l)] * dt
        return rng.standard_normal(rate.shape) * self._noise(hyperparam) * np.sqrt(dt) + rate

    @_on_device
    def m_step(self, param_curr, y, log_posterior_curr, tuning_basis, hyperparam, opt_state_curr=None):
        """reference core.py:895-902: sufficient statistics + the analytic solve."""
        y_dev = self._dev(_unwrap_tsd(y)[0])
        post = torch.exp(self._dev(log_posterior_curr))
        yw = ops.atb(post, y_dev)
        tw = post.sum(dim=0, dtype=torch.float64).to(torch.float32)
        W = self._dev(param_curr).clone()
        self._mstep_fn(hyperparam)(self._dev(tuning_basis), yw, tw, W)
        return {'params': self._host(W), 'opt_state': None}


class GaussianGPLVMJump1D(_GaussianMixin, PoissonGPLVMJump1D):
    """Gaussian GPLVM with jumps (reference core.py:852-916): same API and result keys as the Poisson jump model."""

    def __init__(self, n_neuron, noise_std=0.5, **kwargs):
        self.noise_std = noise_std
        super().__init__(n_neuron, **kwargs)

    def initialize_params(self, key):
        params, _ = super().initialize_params(key)
        self.tuning = self._init_tuning(params)
        return self.params, self.tuning

    def fit_em(self, y, hyperparam={}, key=0, n_iter=20, log_posterior_init=None, ma_neuron=None, ma_latent=None,
               n_time_per_chunk=10000, dt=1., likelihood_scale=1., save_every=None, **kwargs):
        hp = dict(hyperparam)
        hp['noise_std'] = hp.get('noise_std', self.noise_std)
        em = super().fit_em(y, hyperparam=hp, key=key, n_iter=n_iter, log_posterior_init=log_posterior_init,
                            ma_neuron=ma_neuron, ma_latent=ma_latent, n_time_per_chunk=n_time_per_chunk, dt=dt,
                            likelihood_scale=likelihood_scale, save_every=save_every, **kwargs)
        em['m_step_res_l'] = {'params': [], 'opt_state': []}        # reference core.py:654-658 with its m_step dict
        return em


# ------------------------------------------------------------------------------------------------------------
# latent-only families
# ------------------------------------------------------------------------------------------------------------
class _GPLVM1DBase(PoissonGPLVMJump1D):
    """``AbstractGPLVM1D`` (reference core.py:76-373) on the jump kernels with a degenerate dynamics chain."""

    def __init__(self, n_neuron, n_latent_bin=100, tuning_lengthscale=5., param_prior_std=1.,
                 movement_variance=1., explained_variance_threshold_basis=0.999,
                 rng_init_int=123, w_init_variance=1., w_init_mean=0., basis_type='rbf', custom_tuning_kernel=None,
                 custom_transition_kernel=None, smoothness_penalty=0., device=None):
        super().__init__(n_neuron, n_latent_bin=n_latent_bin, tuning_lengthscale=tuning_lengthscale,
                         param_prior_std=param_prior_std, movement_variance=movement_variance,
                         explained_variance_threshold_basis=explained_variance_threshold_basis,
                         rng_init_int=rng_init_int, w_init_variance=w_init_variance, w_init_mean=w_init_mean,
                         p_move_to_jump=0., p_jump_to_move=0., basis_type=basis_type,
                         custom_tuning_kernel=custom_tuning_kernel, custom_transition_kernel=custom_transition_kernel,
                         smoothness_penalty=smoothness_penalty, device=device)
        self.custom_tuning_kernel = custom_tuning_kernel
        del self.p_move_to_jump, self.p_jump_to_move, self.possible_dynamics

    def _init_tuning(self, params):
        return np.logaddexp(self.tuning_basis @ params, np.float32(0)).astype(np.float32)

    def initialize_params(self, key):
        """reference core.py:120-126 (no w_init_mean in the latent-only base class)."""
        params = (jaxprng.normal(key, (self.n_basis, self.n_neuron))
                  * np.float32(np.sqrt(self.w_init_variance))).astype(np.float32)
        self.params = params
        self.tuning = self._init_tuning(params)
        return self.params, self.tuning

    def init_latent_posterior(self, T, key, random_scale=0.1):
        """reference core.py:238-247: (1/K + uniform * random_scale), row normalised."""
        K = self.n_latent_bin
        post = np.float32(1.0 / K) + jaxprng.uniform(key, (T, K)) * np.float32(random_scale)
        post = (post / post.sum(axis=1, keepdims=True)).astype(np.float32)
        return np.log(post), post

    # -- degenerate dynamics: M = identity, all mass on the "move" state
    def _transition_pack(self, hyperparam):
        mv = hyperparam.get('movement_variance', self.movement_variance)
        ck = self.custom_transition_kernel
        ck_key = None if ck is None else hash(np.ascontiguousarray(np.asarray(ck, dtype=np.float32)).tobytes())
        key = (float(mv), ck_key, self.n_latent_bin, str(self.device))
        cached = getattr(self, "_pack_cache", None)
        if cached is not None and cached[0] == key:
            return cached[1]
        K = self.n_latent_bin
        P, logP, _, _ = gpk.create_transition_prob_1d(self.possible_latent_bin, None, mv, 0., 0., custom_kernel=ck)
        M = np.eye(2, dtype=np.float32)
        with np.errstate(divide="ignore"):
            logM = np.log(M)
        host = gpk.move_operator_host(K, mv, ck, p_move_to_jump=None)
        op = ops.MoveOperator(host, M, self.device, P0=None)
        start = np.zeros((2, K), np.float32)
        start[0] = 1.0 / K                              # uniform over the latent (decoder_latentonly.py:66-68)
        op.stationary = torch.from_numpy(start).to(self.device)
        self._pack_cache = (key, (P, logP, M, logM, op))
        return P, logP, M, logM, op

    def _estep(self, y_dev, hyperparam, ma_neuron, ma_latent, likelihood_scale):
        P, logP, M, logM, op = self._transition_pack(hyperparam)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, y_dev.shape[0])
        es = EStep(y_dev, op, ma_n, ma_l, likelihood_scale, emission_factory=self._emission_factory(hyperparam),
                   carry_in=op.stationary)
        return es, logP

    _underflow_msg = ("latent-only filter: the one-step predictive probability underflowed (an observation lies "
                      "where the smooth prior is zero in fp32); use the jump model for such data")

    @classmethod
    def _finite(cls, lml):
        v = float(lml)
        if not np.isfinite(v):
            raise RuntimeError(cls._underflow_msg)
        return v

    @_on_device
    def _decode_latent(self, y, tuning, hyperparam, log_latent_transition_kernel=None, ma_neuron=None,
                       ma_latent=None, likelihood_scale=1., n_time_per_chunk=10000, return_device=False):
        """reference core.py:946-957 / decoder_latentonly.py:150-226: the 6-tuple without the dynamics axis
        (log_acausal_posterior_all [T,K], log_marginal_final, log_causal_posterior_all [T,K],
        log_one_step_predictive_marginals [T], log_accumulated_joint_total [K,K], log_likelihood_all [T,K])."""
        y_dev = self._dev(_unwrap_tsd(y)[0])
        es, logP = self._estep(y_dev, hyperparam, ma_neuron, ma_latent, likelihood_scale)
        T, K = y_dev.shape[0], self.n_latent_bin
        res = es.run(self._dev(tuning), want_gamma=False, want_gamma_lat=True, want_dyn=False, want_r=T > 1)
        self._finite(res.log_marginal)
        log_acc = None
        if T > 1:
            c = res.core
            A = res.alpha_ext.view(-1, 2 * K)[c.start:c.stop - 1, :K]
            R = res.r_ext.view(-1, 2 * K)[c.start + 1:c.stop, :K]
            G = ops.atb_bf16x2(A, R) if T - 1 >= ops.XI_TC_MIN_BINS else ops.atb(A, R)
            log_acc = self._dev(logP[0]) + torch.log(G)              # decoder_latentonly.py:118-131
        out = (torch.log(res.gamma_lat), res.log_marginal.to(torch.float32), torch.log(res.alpha[:, 0, :]),
               res.lmr, log_acc, res.ll)
        if return_device:
            return out
        return tuple(None if o is None else self._host(o) for o in out)

    @_on_device
    def decode_latent(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None, likelihood_scale=1.,
                      n_time_per_chunk=10000, t_l=None):
        """reference core.py:137-178 (keys: log_posterior_all, log_marginal_final, posterior_all,
        log_one_step_predictive_marginals_all, log_likelihood_all, p_/log_ joint_/transition_latent)."""
        y, t_in = _unwrap_tsd(y)
        if t_in is not None:
            t_l = t_in
        if tuning is None:
            tuning = self.tuning
        tup = self._decode_latent(y, tuning, dict(hyperparam), None, ma_neuron, ma_latent, likelihood_scale,
                                  n_time_per_chunk, return_device=True)
        log_post, lml, _, lmr, log_acc, ll = tup
        res = {'log_posterior_all': self._host(log_post),
               'log_marginal_final': float(lml.item()),
               'posterior_all': _rewrap_tsd(self._host(torch.exp(log_post)), t_l),
               'log_one_step_predictive_marginals_all': hostio.LazyHostArray(lmr),
               'log_likelihood_all': self._host(ll)}
        if log_acc is not None:
            lse = torch.logsumexp
            log_joint = log_acc - lse(log_acc.reshape(-1), 0)        # decoder_latentonly.py:229-248
            log_trans = log_joint - lse(log_joint, dim=1, keepdim=True)
            lazy = hostio.LazyHostArray
            res.update({'p_joint_latent': lazy(torch.exp(log_joint)), 'p_transition_latent': lazy(torch.exp(log_trans)),
                        'log_joint_latent': lazy(log_joint), 'log_transition_latent': lazy(log_trans)})
        return res

    @_on_device
    def decode_latent_viterbi(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None,
                              likelihood_scale=1., n_time_per_chunk=10000, t_l=None, return_device=False,
                              time_sharded=False, group=None):
        """Most probable latent path argmax p(x_0..x_{T-1}, y) (beyond the reference): the jump model's Viterbi
        decoding with the degenerate dynamics chain, starting from the uniform latent prior of decode_latent.
        Returns ``map_latent`` (int64 [T]) and ``log_joint_map``; no ``map_dynamics``.  A bin whose normaliser
        underflows raises RuntimeError, as in decode_latent (time-sharded: on every rank, decided from all-reduced
        data).  time_sharded / group: as in PoissonGPLVMJump1D.decode_latent_viterbi."""
        y, t_in = _unwrap_tsd(y)
        if t_in is not None:
            t_l = t_in
        try:
            path, lj = self._viterbi(y, tuning, hyperparam, ma_neuron, ma_latent, likelihood_scale,
                                     lambda op: op.stationary, time_sharded, group)
        except viterbi.SeamError as e:      # an underflowed message never matches its neighbour's
            raise RuntimeError(str(e) + "; " + self._underflow_msg) from e
        self._finite(lj)
        conv = (lambda t: t) if return_device else self._host
        return {'map_latent': _rewrap_tsd_1d(conv(path % self.n_latent_bin), t_l), 'log_joint_map': lj}

    def sample_latent(self, T, key=0, movement_variance=1, init_latent=None):
        """reference core.py:206-227 (NumPy stream)."""
        rng = np.random.default_rng(_seed_from_key(key))
        P, _, _, _ = gpk.create_transition_prob_1d(self.possible_latent_bin, None, movement_variance, 0., 0.,
                                                   custom_kernel=self.custom_transition_kernel)
        P0 = P[0].astype(np.float64)
        P0 /= P0.sum(axis=1, keepdims=True)
        x = int(rng.integers(0, self.n_latent_bin)) if init_latent is None else int(init_latent)
        out = np.empty(T, dtype=np.int64)
        for t in range(T):
            x = int(rng.choice(self.n_latent_bin, p=P0[x]))
            out[t] = x
        return out

    def sample(self, T, hyperparam={}, key=0, init_latent=None, dt=1., tuning=None):
        """reference core.py:229-236."""
        seed = _seed_from_key(key)
        mv = hyperparam.get('movement_variance', self.movement_variance)
        latent_l = self.sample_latent(T, seed, mv, init_latent)
        return latent_l, self.sample_y(latent_l, hyperparam, tuning, dt, seed + 1)

    @_on_device
    def fit_em(self, y, hyperparam={}, key=0, n_iter=20, log_posterior_init=None, opt_state_curr=None,
               ma_neuron=None, ma_latent=None, n_time_per_chunk=10000, dt=1., likelihood_scale=1., save_every=None,
               m_step_step_size=0.01, m_step_maxiter=1000, m_step_tol=1e-6,
               posterior_init_kwargs={'random_scale': 0.1}, verboase=True, **kwargs):
        """reference core.py:256-373 (+ :995-1016 / :1083-1093): M-step, tuning, E-step per iteration; em_res keys as
        there (posterior [T,K], no dynamics marginals)."""
        y_in, t_l = _unwrap_tsd(y)
        hp = dict(hyperparam)
        hp['param_prior_std'] = hp.get('param_prior_std', self.param_prior_std)
        self.tuning_lengthscale = hp.get('tuning_lengthscale', self.tuning_lengthscale)
        self.movement_variance = hp.get('movement_variance', self.movement_variance)
        T, K = int(np.shape(y_in)[0]), self.n_latent_bin
        y_dev = self._dev(y_in)
        if save_every is None:
            save_every = n_iter
        P, logP, M, logM, op = self._transition_pack(hp)
        ma_n, ma_l = self._masks(ma_neuron, ma_latent, T)
        if 'tuning_lengthscale' in hyperparam:
            tuning_basis = gpk.generate_basis(self.tuning_lengthscale, K, self.explained_variance_threshold_basis,
                                              include_bias=True, basis_type=self.basis_type,
                                              custom_kernel=self.custom_tuning_kernel)
        else:
            tuning_basis = self.tuning_basis
        if log_posterior_init is None:
            log_posterior_init, _ = self.init_latent_posterior(T, jaxprng.as_key(key),
                                                               posterior_init_kwargs.get('random_scale', 0.1))
        mstep_fn = self._mstep_fn(hp)
        loop = EMLoop(self, y_dev, op, ma_n, ma_l, likelihood_scale, tuning_basis, log_posterior_init,
                      hp['param_prior_std'], m_step_step_size, m_step_maxiter, m_step_tol,
                      emission_factory=self._emission_factory(hp), carry_in=op.stationary, mstep_fn=mstep_fn)
        self.opt_state_init_fun = ops.AdamState
        saved = {'log_posterior_all_saved': [], 'params_saved': [], 'tuning_saved': [], 'iter_saved': [],
                 'log_marginal_saved': []}
        lml_l, m_hist = [], []
        res = tuning = None
        for i in range(n_iter):
            last, snap = i == n_iter - 1, (i % save_every == 0)
            res, m_res = loop.iteration(want_gamma_lat=(last or snap), speculate=not last)
            m_hist.append(m_res)
            tuning = m_res[4]
            lml_l.append(self._finite(res.log_marginal))
            if snap:
                saved['log_posterior_all_saved'].append(hostio.LazyHostArray(res.gamma_lat, torch.log))
                saved['params_saved'].append(self._host(loop.W_iter.clone()))
                saved['tuning_saved'].append(self._host(tuning))
                saved['log_marginal_saved'].append(np.float32(lml_l[-1]))
                saved['iter_saved'].append(i)
        if mstep_fn is None and m_hist:
            n_its = torch.cat([h[2] for h in m_hist]).cpu().numpy()
            m_step_res_l = {'n_iter': [int(n) for n in n_its],
                            'final_loss': [float(h[3][0].item()) for h in m_hist],
                            'final_error': [float(h[3][1].item()) for h in m_hist],
                            'loss_history': [self._host(h[0][:int(n)]) for h, n in zip(m_hist, n_its)],
                            'error_history': [self._host(h[1][:int(n)]) for h, n in zip(m_hist, n_its)]}
        else:
            m_step_res_l = {'params': [], 'opt_state': []} if mstep_fn is not None else {}
        self.params = self._host(loop.W)
        if n_iter > 0:
            self.tuning = self._host(tuning)
            self.log_marginal_final = np.float32(lml_l[-1])
        self.log_latent_transition_kernel = logP[0]
        self.tuning_basis = tuning_basis
        self._opt_state = loop.state
        self._last_estep_info = {"n_chain": loop.es.plan.n_chain, "chunk_len": loop.es.chunk_len,
                                 "tensor_core_statistics": bool(loop.use_tc),
                                 "compact_scan": bool(loop.es.compact_ok and loop.use_tc)}
        em_res = dict(saved)
        em_res.update({'log_posterior_init': log_posterior_init, 'params': self.params, 'tuning': self.tuning,
                       'log_marginal_l': [np.float32(v) for v in lml_l], 'm_step_res_l': m_step_res_l})
        if n_iter > 0:
            em_res.update({'log_posterior_final': hostio.LazyHostArray(res.gamma_lat, torch.log),
                           'log_marginal': np.float32(lml_l[-1]),
                           'posterior': _rewrap_tsd(self._host(res.gamma_lat), t_l)})
        return em_res


class PoissonGPLVM1D(_GPLVM1DBase):
    """Poisson GPLVM with a smooth latent only, no dynamics (reference core.py:919-1019)."""


class GaussianGPLVM1D(_GaussianMixin, _GPLVM1DBase):
    """Gaussian GPLVM with a smooth latent only (reference core.py:1022-1093)."""

    def __init__(self, n_neuron, noise_std=0.5, **kwargs):
        self.noise_std = noise_std
        super().__init__(n_neuron, **kwargs)

    def decode_latent(self, y, tuning=None, hyperparam={}, **kw):
        hp = dict(hyperparam)
        hp['noise_std'] = hp.get('noise_std', self.noise_std)
        return super().decode_latent(y, tuning=tuning, hyperparam=hp, **kw)
