"""NumPy restatement of the reference's EM hot path (TEST INFRASTRUCTURE ONLY).

Pinned against the reference's own source files run on ``oracle/jaxshim`` (golden vectors in
``tests/golden``; what that does and does not cover: ``oracle/__init__.py``).  Every function names the reference
lines it restates (paths relative to ``/root/reference/poor_man_gplvm/``).  The
arithmetic follows the reference's *operation order* (log space, one
``logsumexp`` per reduction, per-step ``[2,2,K,K]`` joint in the smoother) so
that ``dtype=np.float32`` mimics the JAX fp32 run and ``dtype=np.float64`` is the
ground truth used to arbitrate between two fp32 implementations.

Third-party semantics restated from jax 0.4.26 / optax 0.2.2 (not vendored in
the reference; pinned only in its README.md:25,61):
  * ``logsumexp``: max-shift with non-finite max replaced by 0.
  * ``logaddexp(a,b) = max + log1p(exp(-|a-b|))``.
  * ``softplus(x) = logaddexp(x, 0)``; ``xlogy(0, y) = 0``.
  * ``norm.logpdf(x,0,s) = -(log(2 pi s^2) + x^2/s^2)/2``.
  * ``optax.adam``: bias-corrected, eps outside the sqrt, eps_root = 0.
"""
from __future__ import annotations

import math

import numpy as np
from scipy.special import gammaln

VERY_NEG_LL = -1e20      # decoder.py:46
ACC_INIT = -1e40         # decoder.py:240 (overflows to -inf in fp32, as in the reference)


# ----------------------------------------------------------------------------
# small primitives (jax.scipy.special semantics)
# ----------------------------------------------------------------------------
def lse(a, axis=None, keepdims=False):
    a = np.asarray(a)
    m = np.max(a, axis=axis, keepdims=True)
    m = np.where(np.isfinite(m), m, 0).astype(a.dtype)
    with np.errstate(divide="ignore"):
        out = np.log(np.sum(np.exp(a - m), axis=axis, keepdims=True)) + m
    if not keepdims:
        out = np.squeeze(out, axis=axis) if axis is not None else out.reshape(())
    return out.astype(a.dtype)


def logaddexp(a, b):
    with np.errstate(invalid="ignore"):
        return np.logaddexp(a, b)


def softplus(x):
    return np.logaddexp(x, np.zeros((), dtype=x.dtype))


def xlogy(x, y):
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(x == 0, np.zeros((), dtype=y.dtype), x * np.log(y))


# ----------------------------------------------------------------------------
# gp_kernel.py
# ----------------------------------------------------------------------------
def create_transition_prob_1d(n_latent_bin, movement_variance=1.0, p_move_to_jump=0.01,
                              p_jump_to_move=0.01, custom_kernel=None, dtype=np.float32):
    """gp_kernel.py:42-89 (rbf_kernel :14-20, uniform_kernel :36-40,
    discrete_transition_kernel :30-34).

    Returns (P[2,K,K], logP[2,K,K], M[2,2], logM[2,2]); P[d'][x, x'] is the
    probability of x -> x' under *next* dynamics d'.  The RBF log kernel is
    analytic (finite where the linear one underflows, :19,:79); the exponent is
    -(x-x')^2 / mv^2 with no factor 1/2 (:17).
    """
    K = int(n_latent_bin)
    x = np.arange(K).astype(dtype)
    if custom_kernel is None:
        d2 = (x[:, None] - x[None, :]) ** 2
        mv = dtype(movement_variance)
        lin0 = np.exp(-d2 / mv ** 2) * dtype(1.0)
        log0 = -d2 / mv ** 2 + np.log(dtype(1.0))
    else:
        lin0 = np.asarray(custom_kernel, dtype=dtype)
        with np.errstate(divide="ignore"):
            log0 = np.log(lin0)
        log0 = np.where(log0 == np.inf, dtype(-10000.0), log0)   # get_log, :9-12
    lin1 = np.full((K, K), dtype(1.0) / dtype(K), dtype=dtype)
    log1 = np.log(lin1)
    P, logP = [], []
    for lin, lg in ((lin0, log0), (lin1, log1)):
        z = lin.sum(axis=1, keepdims=True)
        P.append(lin / z)
        logP.append(lg - np.log(z))
    M = np.array([[1 - p_move_to_jump, p_move_to_jump],
                  [p_jump_to_move, 1 - p_jump_to_move]], dtype=dtype)
    with np.errstate(divide="ignore"):
        logM = np.log(M)
    return (np.stack(P).astype(dtype), np.stack(logP).astype(dtype), M, logM.astype(dtype))


# ----------------------------------------------------------------------------
# core.py:41-73
# ----------------------------------------------------------------------------
def generate_basis(lengthscale, n_latent_bin, explained_variance_threshold_basis=0.999,
                   include_bias=True, custom_kernel=None, dtype=np.float32):
    """core.py:41-73: RBF Gram -> SVD -> keep columns until the cumulative
    singular-value fraction crosses the threshold, scale by S^(1/4), prepend 1s."""
    K = int(n_latent_bin)
    if custom_kernel is None:
        x = np.arange(K).astype(dtype)
        gram = np.exp(-((x[:, None] - x[None, :]) ** 2) / dtype(lengthscale) ** 2)
    else:
        gram = np.asarray(custom_kernel, dtype=dtype)
    U, S, _ = np.linalg.svd(gram.astype(dtype))
    n_basis = int((np.cumsum(S / S.sum()) < explained_variance_threshold_basis).sum()) + 1
    basis = U[:, :n_basis] * np.sqrt(np.sqrt(S))[:n_basis][None, :]
    if include_bias:
        basis = np.concatenate([np.ones((K, 1), dtype=dtype), basis.astype(dtype)], axis=1)
    return basis.astype(dtype)


# ----------------------------------------------------------------------------
# fit_tuning_helper.py
# ----------------------------------------------------------------------------
def get_tuning_softplus(params, basis):
    """fit_tuning_helper.py:11-25."""
    return softplus(basis @ params)


def get_statistics(log_posterior_probs, y):
    """fit_tuning_helper.py:28-42."""
    post = np.exp(log_posterior_probs)
    return post.T @ y.astype(post.dtype), post.sum(axis=0)


def poisson_m_step_objective(param, param_prior_std, basis, y_weighted, t_weighted):
    """fit_tuning_helper.py:63-81 (prior constants included in the loss)."""
    dt = param.dtype
    pf = get_tuning_softplus(param, basis)
    norm_term = pf * t_weighted[:, None]
    fit_term = xlogy(y_weighted, pf + dt.type(1e-20))
    log_like = np.sum(fit_term - norm_term)
    s = dt.type(param_prior_std)
    log_prior = np.sum(-(np.log(dt.type(2 * math.pi) * s * s) + param * param / (s * s)) / dt.type(2))
    return -log_like - log_prior


def poisson_m_step_value_and_grad(param, param_prior_std, basis, y_weighted, t_weighted):
    """Hand gradient of the objective above (jax.value_and_grad at
    fit_tuning_helper.py:140,168): dL/dW = -Phi^T[(yw/(pf+1e-20) - tw) * sigmoid(Phi W)] + W/s^2."""
    dt = param.dtype
    z = basis @ param
    pf = softplus(z)
    sig = dt.type(1) / (dt.type(1) + np.exp(-z))
    e = (y_weighted / (pf + dt.type(1e-20)) - t_weighted[:, None]) * sig
    s = dt.type(param_prior_std)
    grad = -(basis.T @ e) + param / (s * s)
    loss = poisson_m_step_objective(param, param_prior_std, basis, y_weighted, t_weighted)
    return loss, grad.astype(dt)


def adam_init(params):
    """optax.adam(...).init (fit_tuning_helper.py:131-132): count=0, mu=0, nu=0."""
    return {"count": 0, "mu": np.zeros_like(params), "nu": np.zeros_like(params)}


def adam_run(params, opt_state, param_prior_std, basis, y_weighted, t_weighted,
             step_size=0.01, maxiter=1000, tol=1e-6, b1=0.9, b2=0.999, eps=1e-8, min_iters=5):
    """fit_tuning_helper.py:124-196 (make_adam_runner.run).

    Loop carried state (i, params, opt_state, error, loss, loss_prev); body runs
    while ``i < maxiter-1 and (i < min_iters or |loss-loss_prev|/max(|loss|,1e-8) > tol)``;
    ``loss`` lags ``params`` by one update (:168-179).  The reference hard-codes
    ``min_iters = 5``; the M-step kernels take it as an argument.
    """
    dt = params.dtype
    f = dt.type
    loss, g = poisson_m_step_value_and_grad(params, param_prior_std, basis, y_weighted, t_weighted)
    err = np.sqrt(np.sum(np.square(g)))
    loss_hist = np.zeros(maxiter, dtype=dt)
    err_hist = np.zeros(maxiter, dtype=dt)
    loss_hist[0], err_hist[0] = loss, err
    i, loss_prev = 0, loss
    count, mu, nu = int(opt_state["count"]), opt_state["mu"].copy(), opt_state["nu"].copy()
    while True:
        rel = abs(loss - loss_prev) / max(abs(loss), f(1e-8))
        if not (i < maxiter - 1 and (i < min_iters or rel > f(tol))):
            break
        new_loss, g = poisson_m_step_value_and_grad(params, param_prior_std, basis, y_weighted, t_weighted)
        mu = f(b1) * mu + f(1 - b1) * g
        nu = f(b2) * nu + f(1 - b2) * (g * g)
        count += 1
        mu_hat = mu / f(1 - f(b1) ** count)
        nu_hat = nu / f(1 - f(b2) ** count)
        params = params + f(-step_size) * (mu_hat / (np.sqrt(nu_hat) + f(eps)))
        err = np.sqrt(np.sum(np.square(g)))
        i += 1
        loss_hist[i], err_hist[i] = new_loss, err
        loss_prev, loss = loss, new_loss
    return {"params": params.astype(dt), "opt_state": {"count": count, "mu": mu, "nu": nu},
            "n_iter": i + 1, "final_loss": loss, "final_error": err,
            "loss_history": loss_hist, "error_history": err_hist}


# ----------------------------------------------------------------------------
# decoder.py — emission and naive Bayes
# ----------------------------------------------------------------------------
def get_loglikelihood_ma_all(y_l, tuning, ma_neuron, ma_latent, dt_l=1.0):
    """decoder.py:30-48 vmapped as :60-85.  ``ma_neuron`` is [N] or [T,N]."""
    fd = tuning.dtype
    T = y_l.shape[0]
    y = y_l.astype(fd)
    ma_n = np.broadcast_to(np.asarray(ma_neuron, dtype=fd), y.shape)
    dt_b = np.broadcast_to(np.asarray(dt_l, dtype=fd), (T,))
    out = np.empty((T, tuning.shape[0]), dtype=fd)
    lg = gammaln(y + fd.type(1.0)).astype(fd)
    step = max(1, int(4e6 // max(1, tuning.size)))
    for s in range(0, T, step):
        e = min(T, s + step)
        lam = tuning[None, :, :] * dt_b[s:e, None, None] + fd.type(1e-20)     # [t,K,N]
        ll = xlogy(y[s:e, None, :], lam) - lam - lg[s:e, None, :]
        out[s:e] = (ll * ma_n[s:e, None, :]).sum(axis=2)
    return np.where(np.asarray(ma_latent).astype(bool)[None, :], out, fd.type(VERY_NEG_LL))


def get_naive_bayes_ma_chunk(y, tuning, ma_neuron, ma_latent, dt_l=1.0, n_time_per_chunk=10000):
    """decoder.py:88-149."""
    T = y.shape[0]
    fd = tuning.dtype
    ma_n = np.broadcast_to(np.asarray(ma_neuron, dtype=fd), y.shape)
    dt_b = np.broadcast_to(np.asarray(dt_l, dtype=fd), (T,))
    posts, lmls, tot, lls = [], [], [], []
    for s in range(0, T, n_time_per_chunk):
        sl = slice(s, s + n_time_per_chunk)
        ll = get_loglikelihood_ma_all(y[sl], tuning, ma_n[sl], ma_latent, dt_b[sl])
        lml = lse(ll, axis=-1, keepdims=True)
        posts.append(ll - lml)
        lmls.append(lml[:, 0])
        tot.append(np.sum(lml))
        lls.append(ll)
    return (np.concatenate(posts), np.concatenate(lmls),
            np.sum(np.array(tot, dtype=fd)), np.concatenate(lls))


# ----------------------------------------------------------------------------
# decoder.py — forward filter / backward smoother
# ----------------------------------------------------------------------------
def filter_one_step(post_prev, lml_prev, ll_curr, logP, logM, likelihood_scale=1.0):
    """decoder.py:151-172."""
    a = lse(post_prev[:, None, :] + logM[:, :, None], axis=0)      # [d', x]
    prior = lse(a[:, :, None] + logP, axis=1)                      # [d', x']
    u = prior + ll_curr.dtype.type(likelihood_scale) * ll_curr[None, :]
    lmr = lse(u)
    return u - lmr, lml_prev + lmr, prior, lmr


def filter_all_step(ll_all, logP, logM, carry_init=None, likelihood_scale=1.0):
    """decoder.py:174-187.  Initial carry: uniform over the joint state, lml 0."""
    fd = ll_all.dtype
    K, D = logP.shape[1], logM.shape[0]
    if carry_init is None:
        post = np.log(np.ones((D, K), dtype=fd) / fd.type(D * K))
        lml = fd.type(0)
    else:
        post, lml = carry_init
    T = ll_all.shape[0]
    posts = np.empty((T, D, K), dtype=fd)
    priors = np.empty((T, D, K), dtype=fd)
    lmrs = np.empty((T,), dtype=fd)
    for t in range(T):
        post, lml, prior, lmr = filter_one_step(post, lml, ll_all[t], logP, logM, likelihood_scale)
        posts[t], priors[t], lmrs[t] = post, prior, lmr
    return posts, lml, priors, lmrs


def smooth_one_step(s_next, acc, f_curr, prior_next, logP, logM, accumulate=True):
    """decoder.py:200-226.  joint[d, d', x, x']."""
    diff = s_next - prior_next
    joint = (logP[None, :, :, :] + logM[:, :, None, None]
             + diff[None, :, None, :] + f_curr[:, None, :, None])
    s_curr = lse(joint, axis=(1, 3))
    if accumulate:
        acc = logaddexp(acc, joint)
    return s_curr, acc


def smooth_all_step(f_all, prior_all, logP, logM, carry_init=None, accumulate=True):
    """decoder.py:230-256 (reverse scan; last chunk starts from the filtered
    posterior of the final bin and an all ``-1e40`` accumulator)."""
    fd = f_all.dtype
    D, K = f_all.shape[1], f_all.shape[2]
    n = f_all.shape[0]
    out = np.empty_like(f_all)
    if carry_init is None:
        s = f_all[-1]
        with np.errstate(over="ignore"):
            acc = (np.ones((D, D, K, K), dtype=fd) * fd.type(ACC_INIT)) if accumulate else None
        out[-1] = s
        idx = range(n - 2, -1, -1)
    else:
        s, acc = carry_init
        idx = range(n - 1, -1, -1)
    # prior_all[j] pairs with f_all[j] and is the causal prior of bin j+1
    for j in idx:
        s, acc = smooth_one_step(s, acc, f_all[j], prior_all[j], logP, logM, accumulate)
        out[j] = s
    return out, acc


def smooth_all_step_combined_ma_chunk(y, tuning, logP, logM, ma_neuron, ma_latent=None,
                                      likelihood_scale=1.0, n_time_per_chunk=10000,
                                      accumulate=True):
    """decoder.py:258-332: chunked forward pass carrying (post_last, lml), then
    chunked backward pass carrying (s_first, acc)."""
    fd = tuning.dtype
    T = y.shape[0]
    if ma_latent is None:
        ma_latent = np.ones(tuning.shape[0], dtype=fd)
    ma_neuron = np.asarray(ma_neuron)
    slices, f_chunks, prior_chunks, lmr_chunks, ll_chunks = [], [], [], [], []
    carry = None
    lml = fd.type(0)
    for s in range(0, T, n_time_per_chunk):
        sl = slice(s, min(T, s + n_time_per_chunk))
        slices.append(sl)
        ma_c = ma_neuron[sl] if ma_neuron.ndim == 2 else ma_neuron
        ll = get_loglikelihood_ma_all(y[sl], tuning, ma_c, ma_latent)
        posts, lml, priors, lmrs = filter_all_step(ll, logP, logM, carry, likelihood_scale)
        carry = (posts[-1], lml)
        f_chunks.append(posts); prior_chunks.append(priors)
        lmr_chunks.append(lmrs); ll_chunks.append(ll)
    prior_cat = np.concatenate(prior_chunks)
    s_chunks = []
    carry_b = None
    for n in range(len(slices) - 1, -1, -1):
        sl = slices[n]
        pri = prior_cat[sl.start + 1: sl.stop + 1]
        out, acc = smooth_all_step(f_chunks[n], pri, logP, logM, carry_b, accumulate)
        carry_b = (out[0], acc)
        s_chunks.append(out)
    s_chunks.reverse()
    return (np.concatenate(s_chunks), lml, np.concatenate(f_chunks),
            np.concatenate(lmr_chunks), acc, np.concatenate(ll_chunks))


def compute_transition_posterior_prob(log_acc):
    """decoder.py:334-375."""
    log_joint_full = log_acc - lse(log_acc)
    log_joint_latent = lse(log_joint_full, axis=(0, 1))
    log_joint_dynamics = lse(log_joint_full, axis=(2, 3))
    log_transition_latent = log_joint_latent - lse(log_joint_latent, axis=1, keepdims=True)
    log_transition_dynamics = log_joint_dynamics - lse(log_joint_dynamics, axis=1, keepdims=True)
    log_transition_full = log_joint_full - lse(log_joint_full, axis=(1, 3), keepdims=True)
    res = {"log_joint_full": log_joint_full, "log_joint_latent": log_joint_latent,
           "log_joint_dynamics": log_joint_dynamics, "log_transition_full": log_transition_full,
           "log_transition_latent": log_transition_latent,
           "log_transition_dynamics": log_transition_dynamics}
    for k in list(res):
        res["p_" + k[4:]] = np.exp(res[k])
    return res


# ----------------------------------------------------------------------------
# core.py — model class (PoissonGPLVMJump1D on AbstractGPLVMJump1D)
# ----------------------------------------------------------------------------
class OraclePoissonGPLVMJump1D:
    """core.py:376-849 restated on NumPy.  PRNG is *not* JAX's threefry: pass
    ``params`` / ``log_posterior_init`` explicitly for parity runs (SURVEY H6/H7)."""

    def __init__(self, n_neuron, n_latent_bin=100, tuning_lengthscale=1.0, param_prior_std=1.0,
                 movement_variance=1.0, explained_variance_threshold_basis=0.999,
                 rng_init_int=123, w_init_variance=1.0, w_init_mean=0.0, p_move_to_jump=0.01,
                 p_jump_to_move=0.01, custom_transition_kernel=None, dtype=np.float32,
                 tuning_basis=None, params=None):
        self.dtype = np.dtype(dtype)
        self.n_neuron, self.n_latent_bin = n_neuron, n_latent_bin
        self.tuning_lengthscale, self.param_prior_std = tuning_lengthscale, param_prior_std
        self.movement_variance = movement_variance
        self.p_move_to_jump, self.p_jump_to_move = p_move_to_jump, p_jump_to_move
        self.explained_variance_threshold_basis = explained_variance_threshold_basis
        self.custom_transition_kernel = custom_transition_kernel
        if tuning_basis is None:
            tuning_basis = generate_basis(tuning_lengthscale, n_latent_bin,
                                          explained_variance_threshold_basis, dtype=self.dtype.type)
        self.tuning_basis = np.asarray(tuning_basis, dtype=self.dtype)
        self.n_basis = self.tuning_basis.shape[1]
        self.ma_neuron_default = np.ones(n_neuron, dtype=self.dtype)
        self.ma_latent_default = np.ones(n_latent_bin, dtype=self.dtype)
        if params is None:   # core.py:429-437 (numpy PRNG, not threefry)
            rng = np.random.default_rng(rng_init_int)
            params = rng.standard_normal((self.n_basis, n_neuron)) * math.sqrt(w_init_variance) + w_init_mean
        self.params = np.asarray(params, dtype=self.dtype)
        self.tuning = get_tuning_softplus(self.params, self.tuning_basis)

    def _transitions(self, hyperparam):
        mv = hyperparam.get("movement_variance", self.movement_variance)
        pmj = hyperparam.get("p_move_to_jump", self.p_move_to_jump)
        pjm = hyperparam.get("p_jump_to_move", self.p_jump_to_move)
        return create_transition_prob_1d(self.n_latent_bin, mv, pmj, pjm,
                                         self.custom_transition_kernel, dtype=self.dtype.type)

    def init_latent_posterior(self, T, seed=0, random_scale=0.1):
        """core.py:571-583 (numpy PRNG)."""
        rng = np.random.default_rng(seed)
        post = (rng.random((T, self.n_latent_bin)) * random_scale).astype(self.dtype)
        post = post / post.sum(axis=1, keepdims=True)
        with np.errstate(divide="ignore"):
            lp = np.log(post)
        return np.where(np.isneginf(lp), self.dtype.type(ACC_INIT), lp), post

    def m_step(self, params, y, log_posterior_curr, tuning_basis, param_prior_std, opt_state,
               step_size, maxiter, tol):
        """core.py:802-827."""
        yw, tw = get_statistics(log_posterior_curr, y)
        res = adam_run(params, opt_state, param_prior_std, tuning_basis, yw, tw,
                       step_size=step_size, maxiter=maxiter, tol=tol)
        n = res["n_iter"]
        res["loss_history"] = res["loss_history"][:n]
        res["error_history"] = res["error_history"][:n]
        return res

    def fit_em(self, y, hyperparam={}, n_iter=20, log_posterior_init=None, ma_neuron=None,
               ma_latent=None, n_time_per_chunk=10000, likelihood_scale=1.0, save_every=None,
               m_step_step_size=0.01, m_step_maxiter=1000, m_step_tol=1e-6, seed=0,
               accumulate=False):
        """core.py:829-849 -> :592-713.  M-step first, then tuning, then E-step."""
        fd = self.dtype
        y_ = np.asarray(y).astype(fd)
        hp = dict(hyperparam)
        prior_std = hp.get("param_prior_std", self.param_prior_std)
        _, logP, _, logM = self._transitions(hp)
        ma_neuron = self.ma_neuron_default if ma_neuron is None else np.asarray(ma_neuron, dtype=fd)
        ma_latent = self.ma_latent_default if ma_latent is None else np.asarray(ma_latent, dtype=fd)
        basis = self.tuning_basis
        if "tuning_lengthscale" in hp:
            basis = generate_basis(hp["tuning_lengthscale"], self.n_latent_bin,
                                   self.explained_variance_threshold_basis, dtype=fd.type)
        if log_posterior_init is None:
            log_posterior_init, _ = self.init_latent_posterior(y_.shape[0], seed)
        log_posterior_init = np.asarray(log_posterior_init, dtype=fd)
        save_every = n_iter if save_every is None else save_every
        opt_state = adam_init(self.params)
        params, lp_curr = self.params, log_posterior_init
        lml_l, m_hist = [], {}
        saved = {"log_posterior_all_saved": [], "params_saved": [], "tuning_saved": [],
                 "iter_saved": [], "log_marginal_saved": []}
        for i in range(n_iter):
            m_res = self.m_step(params, y_, lp_curr, basis, prior_std, opt_state,
                                m_step_step_size, m_step_maxiter, m_step_tol)
            for k, v in m_res.items():
                if k not in ("params", "opt_state"):
                    m_hist.setdefault(k, []).append(v)
            params, opt_state = m_res["params"], m_res["opt_state"]
            tuning = get_tuning_softplus(params, basis)
            (lp_all, lml, lf_all, lmr_all, acc, ll_all) = smooth_all_step_combined_ma_chunk(
                y_, tuning, logP, logM, ma_neuron, ma_latent, likelihood_scale,
                n_time_per_chunk, accumulate=accumulate)
            lp_curr = lse(lp_all, axis=1)
            lml_l.append(lml)
            if i % save_every == 0:
                saved["log_posterior_all_saved"].append(lp_all)
                saved["params_saved"].append(params); saved["tuning_saved"].append(tuning)
                saved["log_marginal_saved"].append(lml); saved["iter_saved"].append(i)
        self.params, self.tuning, self.log_marginal_final = params, tuning, lml
        self.tuning_basis = basis
        post = np.exp(lp_all)
        res = dict(saved)
        res.update({"log_posterior_init": log_posterior_init, "params": params, "tuning": tuning,
                    "log_posterior_final": lp_all, "log_marginal": lml, "log_marginal_l": lml_l,
                    "posterior": post, "posterior_latent_marg": post.sum(axis=1),
                    "posterior_dynamics_marg": post.sum(axis=2), "m_step_res_l": m_hist,
                    "opt_state": opt_state})
        return res

    def decode_latent(self, y, tuning=None, hyperparam={}, ma_neuron=None, ma_latent=None,
                      likelihood_scale=1.0, n_time_per_chunk=10000):
        """core.py:454-497."""
        fd = self.dtype
        tuning = self.tuning if tuning is None else np.asarray(tuning, dtype=fd)
        ma_neuron = self.ma_neuron_default if ma_neuron is None else np.asarray(ma_neuron, dtype=fd)
        ma_latent = self.ma_latent_default if ma_latent is None else np.asarray(ma_latent, dtype=fd)
        _, logP, _, logM = self._transitions(hyperparam)
        (lp_all, lml, lf_all, lmr_all, acc, ll_all) = smooth_all_step_combined_ma_chunk(
            np.asarray(y).astype(fd), tuning, logP, logM, ma_neuron, ma_latent, likelihood_scale,
            n_time_per_chunk, accumulate=True)
        post = np.exp(lp_all)
        res = {"log_posterior_all": lp_all, "log_marginal_final": float(lml), "posterior_all": post,
               "posterior_latent_marg": post.sum(axis=1), "posterior_dynamics_marg": post.sum(axis=2),
               "log_one_step_predictive_marginals_all": lmr_all, "log_likelihood_all": ll_all,
               "log_causal_posterior_all": lf_all, "log_accumulated_joint_total": acc}
        res.update(compute_transition_posterior_prob(acc))
        return res

    def decode_latent_naive_bayes(self, y, tuning=None, ma_neuron=None, ma_latent=None,
                                  n_time_per_chunk=10000, dt_l=1.0):
        """core.py:788-792 -> :499-524."""
        fd = self.dtype
        tuning = self.tuning if tuning is None else np.asarray(tuning, dtype=fd)
        ma_neuron = self.ma_neuron_default if ma_neuron is None else np.asarray(ma_neuron, dtype=fd)
        ma_latent = self.ma_latent_default if ma_latent is None else np.asarray(ma_latent, dtype=fd)
        lp, lml_l, lml_tot, ll = get_naive_bayes_ma_chunk(np.asarray(y).astype(fd), tuning, ma_neuron,
                                                          ma_latent, dt_l, n_time_per_chunk)
        return {"log_posterior_latent": lp, "log_marginal_l": lml_l,
                "log_marginal_total": float(lml_tot), "posterior_latent": np.exp(lp),
                "ll_per_pos_l": ll}
