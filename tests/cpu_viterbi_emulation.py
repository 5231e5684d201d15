"""CPU stand-ins for the Viterbi operators (`csrc/pmg_viterbi.cu`), used ONLY to exercise the host-side
orchestration of `poor_man_gplvm_b200.viterbi.run` -- seam checks, Jacobi repair sweeps, the rank-boundary exchange
and the cross-rank backtrack -- without a GPU, under gloo with several ranks.

They follow the conventions of the kernels they replace (`viterbi_fwd_kernel`, `viterbi_maps_kernel`,
`viterbi_link_kernel`, `viterbi_resolve_kernel` / `viterbi_resolve_sharded_kernel`, `viterbi_fill_kernel`): where a
chain's warm-up starts, what mode 1 restarts from, which message goes to `halo_state` / `end_msg`, the backpointer
layout and the tie rule (smallest flat index), in float64 NumPy.  Test infrastructure: the product path never imports
this module.
"""
from __future__ import annotations

import numpy as np

from cpu_scan_emulation import _chains, _dense_move, _halo_own, _np, _slot


def viterbi_forward(plan, op, ll, bp, lmr, halo_state=None, end_msg=None, carry_in=None, mode=0, chain_ids=None,
                    warm_in=None, warm_out=None, sel_err=None, sel_tol=0.0):
    K = op.K
    P0 = _dense_move(op)
    M = op.M.reshape(2, 2).astype(np.float64)
    scale = float(plan.likelihood_scale)
    ll_, bp_, lmr_ = _np(ll), _np(bp), _np(lmr)
    x = np.arange(K)
    for s, t_begin, t_end in _chains(plan, mode, chain_ids, sel_err, sel_tol):
        msg = None
        if mode != 0:
            t0 = t_begin
            msg = _slot(warm_in, s) if t0 > 0 else (None if carry_in is None else _np(carry_in))
        else:
            t0 = t_begin - _halo_own(plan, s)
            if t0 <= 0 and plan.left_exact:
                t0 = 0
                msg = None if carry_in is None else _np(carry_in)
            else:
                t0 = max(t0, 0)
                msg = None if warm_in is None else _slot(warm_in, s)
        m = None if msg is None else np.array(msg, dtype=np.float64).reshape(2, K)
        tot = 0.0 if m is None else m.sum()
        m = m / tot if (tot > 0 and np.isfinite(tot)) else np.full((2, K), 0.5 / K)
        for t in range(t0, t_end):
            row = ll_[t].astype(np.float64)
            mx = row.max()
            L = np.exp(scale * (row - mx))
            if t == 0:          # the start is marginalised: the filter's prior from the carry
                pr0 = (M[0, 0] * m[0] + M[1, 0] * m[1]) @ P0
                pr1 = (M[0, 1] * m[0].sum() + M[1, 1] * m[1].sum()) / K
                ix0, ix1 = np.zeros(K, np.int64), 0
            else:
                j0 = m[1] * M[1, 0] > m[0] * M[0, 0]
                a0, i0 = np.where(j0, m[1] * M[1, 0], m[0] * M[0, 0]), np.where(j0, K + x, x)
                j1 = m[1] * M[1, 1] > m[0] * M[0, 1]
                a1, i1 = np.where(j1, m[1] * M[1, 1], m[0] * M[0, 1]), np.where(j1, K + x, x)
                pr1 = a1.max()
                ix1 = int(i1[a1 == pr1].min())
                pr1 /= K
                c = a0[:, None] * P0                                    # [x, x']
                pr0 = c.max(axis=0)
                ix0 = np.where(c == pr0[None, :], i0[:, None], 2 * K).min(axis=0)
            u = np.stack([pr0 * L, pr1 * L])
            cn = u.sum()
            m = u / cn
            if t >= t_begin:
                if t > 0:
                    bp_[t, 0, :K] = ix0
                    bp_[t, 1, :K] = ix1
                lmr_[t] = np.float32(np.log(cn) + scale * mx)
            if t == t_begin - 1 and halo_state is not None:
                _np(halo_state)[s] = m.astype(np.float32)
            if t == t_end - 1 and end_msg is not None:
                _np(end_msg)[s] = m.astype(np.float32)


def _bp_at(bp, t, st, K):
    d = int(st >= K)
    return int(bp[t, d, st - d * K])


def _bounds(plan, c):
    b = plan.core_begin + c * plan.chunk_len
    return b, min(b + plan.chunk_len, plan.core_end)


def viterbi_chain_maps(plan, K, bp, maps):
    bp_, maps_ = _np(bp), _np(maps)
    for c in range(plan.n_chain):
        b, e = _bounds(plan, c)
        for s0 in range(2 * K):
            st = s0
            for t in range(e - 1, b, -1):
                st = _bp_at(bp_, t, st, K)
            maps_[c, s0] = st


def _walk_chains(plan, K, bp_, maps_, st, path_, through_begin):
    for c in range(plan.n_chain - 1, -1, -1):
        b, e = _bounds(plan, c)
        if path_ is not None:
            path_[e - 1] = st
        if c > 0 or through_begin:
            st = _bp_at(bp_, b, int(maps_[c, st]), K)
    return st


def _fill(plan, K, bp_, path_):
    for c in range(plan.n_chain):
        b, e = _bounds(plan, c)
        st = int(path_[e - 1])
        for t in range(e - 1, b, -1):
            st = _bp_at(bp_, t, st, K)
            path_[t - 1] = st


def viterbi_block_link(plan, K, bp, maps, link):
    assert plan.core_begin >= 1
    bp_, maps_, link_ = _np(bp), _np(maps), _np(link)
    for s in range(2 * K):
        link_[s] = _walk_chains(plan, K, bp_, maps_, s, None, True)


def viterbi_backtrack(plan, K, bp, maps, last_msg, path):
    bp_, path_ = _np(bp), _np(path)
    _walk_chains(plan, K, bp_, _np(maps), int(np.argmax(_np(last_msg).reshape(-1))), path_, False)
    _fill(plan, K, bp_, path_)


def viterbi_backtrack_sharded(plan, K, bp, maps, gathered, rank, path):
    g = _np(gathered)
    world = g.shape[0]
    st = int(np.argmax(g[world - 1, 2 * K:4 * K].view(np.float32)))
    for r in range(world - 1, rank, -1):
        st = int(g[r, st])
    bp_, path_ = _np(bp), _np(path)
    _walk_chains(plan, K, bp_, _np(maps), st, path_, False)
    _fill(plan, K, bp_, path_)
