"""fp64 log-space Viterbi of the joint (dynamics, latent) chain (TEST INFRASTRUCTURE ONLY).

The reference has no Viterbi decoder, so this is pinned by brute-force enumeration of all paths
(``tests/test_viterbi_cpu.py``) and by its start convention: the log-sum-exp of the path scores is the filter's log
marginal (``linear_ref.forward``).  Conventions of ``PoissonGPLVMJump1D.decode_latent_viterbi``:

* joint state s = d*K + x, transition logM[d,d'] + logP[d'][x,x'] (``gp_kernel.create_transition_prob_1d``);
* bin 0's prior is summed from the carry in front of it (uniform 1/(2K) by default), as in the filter;
* emission likelihood_scale * ll;
* exact ties go to the smallest flat index, in every predecessor max and in the final argmax (among equally good
  paths the decoder returns the one whose states, read from the last bin backwards, are smallest).
"""
from __future__ import annotations

import numpy as np


def start_log_prior(logP, logM, carry=None):
    """log prior [2,K] of bin 0: sum over the carry [2,K] (default uniform) of M[d,d'] P_{d'}[x,x']."""
    logP = np.asarray(logP, dtype=np.float64)
    K = logP.shape[1]
    carry = np.full((2, K), 1.0 / (2 * K)) if carry is None else np.asarray(carry, dtype=np.float64)
    a = np.exp(np.asarray(logM, dtype=np.float64)).T @ carry                  # [d', x]
    with np.errstate(divide="ignore"):
        return np.log(np.stack([a[0] @ np.exp(logP[0]), a[1] @ np.exp(logP[1])]))


def viterbi(ll, logP, logM, likelihood_scale=1.0, carry=None, log_prior0=None, band=None):
    """MAP path of the joint chain.  ll [T,K]; logP [2,K,K]; logM [2,2].  log_prior0 [2,K] overrides the prior from
    the carry.  band: consider only moves with |x - x'| <= band (None = every move: exact).
    Returns (path int64 [T] of flat states d*K + x, log_joint = log p(path, y))."""
    ll = np.asarray(ll, dtype=np.float64)
    T, K = ll.shape
    logP = np.asarray(logP, dtype=np.float64)
    logM = np.asarray(logM, dtype=np.float64)
    e = np.float64(likelihood_scale) * ll
    lp0 = start_log_prior(logP, logM, carry) if log_prior0 is None else np.asarray(log_prior0, dtype=np.float64)
    delta = lp0 + e[0][None, :]
    W = K - 1 if band is None else min(int(band), K - 1)
    # candidates of the move target x': x = x' - W + j, j in [0, 2W]; logP0 gathered per (x', j), -inf outside
    xs = np.arange(K)[:, None] - W + np.arange(2 * W + 1)[None, :]
    inside = (xs >= 0) & (xs < K)
    xc = np.clip(xs, 0, K - 1)
    lp0_band = np.where(inside, logP[0][xc, np.arange(K)[:, None]], -np.inf)          # [x', j]
    bp = np.zeros((T, 2, K), dtype=np.int64)
    rows = np.arange(K)
    for t in range(1, T):
        if band is None:
            # move target: max over every flat predecessor d*K + x (argmax keeps the first, i.e. smallest, index)
            c0 = ((delta + logM[:, 0][:, None])[:, :, None] + logP[0][None]).reshape(2 * K, K)
            k0 = np.argmax(c0, axis=0)
            v0 = c0[k0, rows]
            bp[t, 0] = k0
        else:
            # the same over the band only, d-major (flat index d*K + x increases along d, then along j)
            c0 = delta[:, xc] + logM[:, 0][:, None, None] + lp0_band[None]          # [d, x', j]
            flat = c0.transpose(1, 0, 2).reshape(K, -1)                              # [x', d*(2W+1) + j]
            k0 = np.argmax(flat, axis=1)
            v0 = flat[rows, k0]
            bp[t, 0] = (k0 // (2 * W + 1)) * K + xs[rows, k0 % (2 * W + 1)]
        # jump target: P_1 is constant, one argmax over every (d, x)
        c1 = (delta + logM[:, 1][:, None]).reshape(-1)
        k1 = int(np.argmax(c1))
        v1 = c1[k1] + logP[1][k1 % K, :]
        bp[t, 1] = k1
        delta = np.stack([v0, v1]) + e[t][None, :]
    s = int(np.argmax(delta.reshape(-1)))
    log_joint = float(delta.reshape(-1)[s])
    path = np.empty(T, dtype=np.int64)
    path[T - 1] = s
    for t in range(T - 1, 0, -1):
        s = int(bp[t, s // K, s % K])
        path[t - 1] = s
    return path, log_joint


def score(path, ll, logP, logM, likelihood_scale=1.0, carry=None, log_prior0=None):
    """log p(path, y) of a flat path [T] (states d*K + x) under the same conventions."""
    ll = np.asarray(ll, dtype=np.float64)
    T, K = ll.shape
    logP = np.asarray(logP, dtype=np.float64)
    logM = np.asarray(logM, dtype=np.float64)
    path = np.asarray(path, dtype=np.int64)
    d, x = path // K, path % K
    e = np.float64(likelihood_scale) * ll[np.arange(T), x]
    lp0 = start_log_prior(logP, logM, carry) if log_prior0 is None else np.asarray(log_prior0, dtype=np.float64)
    tr = logM[d[:-1], d[1:]] + logP[d[1:], x[:-1], x[1:]]
    return float(lp0[d[0], x[0]] + e.sum() + tr.sum())
