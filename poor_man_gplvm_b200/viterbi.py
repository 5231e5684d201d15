"""Viterbi decoding: the most probable joint (dynamics, latent) path, time-parallel on the device.

Beyond the reference, which decodes marginals only.  Driven by an ``EStep`` (same emission, chain plan, warm starts
and seam machinery as the filter):

* emission through the E-step's emission operand (any family's ``emission_factory``);
* ``pmg_viterbi_forward`` over all chains, each warming up from the stationary distribution of the prior chain;
  messages are normalised by their sum every bin, so they forget their start geometrically, like the filter's;
* seams (a chain's warmed-up message in front of its first bin against its neighbour's true message there) are
  checked with ``pmg_seam_check_fix``; failed ones are repaired on the device by a conditional relaunch (mode 2),
  and if a seam still fails, by host sweeps that restart the failing chains from their neighbours' messages until
  every seam passes -- the path does not depend on the chunking beyond ``seam_tol``;
* ``pmg_viterbi_chain_maps`` and ``pmg_viterbi_backtrack`` resolve the path, with no host round trip.
"""
from __future__ import annotations

import torch

from . import ops
from .estep import T_FAIL_F, T_FIX_F


class SeamError(RuntimeError):
    """A seam still failed after every repair sweep (e.g. a message that underflowed to zero)."""


class ViterbiResult:
    """path: device int32 [T] of flat states d*K + x; log_joint_map: device fp64 scalar, log p(path, y);
    n_fix / n_relay: seams repaired on the device / by host sweeps; seam_err: worst final seam error."""
    __slots__ = ("path", "log_joint_map", "n_fix", "n_relay", "seam_err", "n_chain")


def run(es, tuning):
    """MAP path of the recording held by ``es`` (a single-device EStep) under ``tuning``."""
    if es.shard.active:
        raise ValueError("Viterbi decoding is not time-sharded")
    S, K, T, dev = es.S, es.K, es.T, es.dev
    K2, tol = 2 * K, es.seam_tol
    plan = es.plan
    plan.halo = plan.halo_next = int(es.halo)
    ops.set_chain_halos(plan)
    ll = es.emission(tuning)
    ops.phase("emission")
    bp = ops.viterbi_bp(T, K, dev)
    # message at the last bin of each chain, one slot ahead: seam c (in front of chain c) finds its truth in slot c
    end_ext = torch.zeros((S + 1, 2, K), dtype=torch.float32, device=dev)
    warm0 = getattr(es.op, "stationary", None)
    tail = es.tail
    tail.zero_()

    def fwd(mode=0, ids=None, **sel):
        ops.viterbi_forward(plan, es.op, ll, bp, es.lmr, halo_state=(es.halo_state if mode == 0 else None),
                            end_msg=end_ext[1:], carry_in=es.carry_in, mode=mode, chain_ids=ids,
                            warm_in=(warm0 if mode == 0 else es.halo_state), **sel)

    def check(fix, slot, err):
        if S > 1:
            ops.seam_check_fix(S - 1, K2, es.halo_state[1].data_ptr(), K2, end_ext[1].data_ptr(), K2, err[1:S], tol,
                               fix, tail[slot:slot + 1])

    def verdict():
        es._verdict_enqueue()
        err, fail, _ = es._verdict_wait()
        return err, fail

    fwd()
    if S > 1 and es.device_repair:
        check(True, T_FIX_F, es.err1)
        fwd(mode=2, sel_err=es.err1[:S], sel_tol=tol)
    check(False, T_FAIL_F, es.err)
    ops.phase("viterbi_forward")
    err, fail = verdict()
    n_fix, n_relay = int(es.tail_host[T_FIX_F]), 0
    for _ in range(es.max_sweeps):
        if not fail:
            break
        bad = torch.nonzero(~(err[1:S] <= tol)).flatten() + 1
        n_relay += int(bad.numel())
        idl = bad.to(dev)
        es.halo_state[idl] = end_ext[idl]                 # restart from the neighbour's current message
        fwd(mode=1, ids=idl.to(torch.int32))
        tail.zero_()
        check(False, T_FAIL_F, es.err)
        err, fail = verdict()
    if fail:
        raise SeamError("Viterbi: seams still above seam_tol=%g after %d repair sweeps (worst %.3g)"
                        % (tol, es.max_sweeps, float(err[1:S].max())))
    maps = torch.empty((S, K2), dtype=torch.int32, device=dev)
    path = torch.empty(T, dtype=torch.int32, device=dev)
    ops.viterbi_chain_maps(plan, K, bp, maps)
    ops.phase("chain_maps")
    ops.viterbi_backtrack(plan, K, bp, maps, end_ext[S], path)
    ops.phase("backtrack")
    res = ViterbiResult()
    res.path = path[es.core]
    res.log_joint_map = es.lmr[es.core].sum(dtype=torch.float64) + torch.log(end_ext[S].max().double())
    res.n_fix, res.n_relay, res.n_chain = n_fix, n_relay, S
    res.seam_err = float(err[1:S].max()) if S > 1 else 0.0
    return res
