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

Time-sharded (an EStep built with ``shard=TimeShard(group)``): the halo rows of y arrive through the E-step's halo
exchange and the forward pass runs unchanged on the rank's extended block.  After it, each rank's last message goes to
the right neighbour (the filter's boundary pack / all-gather / unpack) as the truth of that rank's seam 0, which the
host sweeps repair like any other seam, re-exchanging every sweep; the verdict is all-reduced, so every rank runs the
same sweeps and raises the same errors.  The backtrack then needs ONE all-gather of a fixed-size record per rank
(``pmg_viterbi_block_link``'s map from the block's end state to the left neighbour's, the last message, the partial
sum of lmr), from which ``pmg_viterbi_backtrack_sharded`` resolves every rank's end state on the device.
"""
from __future__ import annotations

import torch

from . import ops
from .estep import T_FAIL_F, T_FIX_F


class SeamError(RuntimeError):
    """A seam still failed after every repair sweep (e.g. a message that underflowed to zero)."""


class ViterbiResult:
    """path: device int32 [T] of flat states d*K + x (this rank's block); log_joint_map: fp64 scalar, log p(path, y)
    (global, identical on every rank); n_fix: seams repaired on the device (all ranks); n_relay: seams of this rank
    repaired by host sweeps, n_relay_boundary of them the rank-boundary seam (chain 0 of a rank > 0);
    seam_err: worst final seam error of this rank."""
    __slots__ = ("path", "log_joint_map", "n_fix", "n_relay", "n_relay_boundary", "seam_err", "n_chain")


def run(es, tuning):
    """MAP path of the recording held by ``es`` under ``tuning``.  On a time-sharded EStep (every rank of the group
    calls this together) the path covers this rank's block and ``log_joint_map`` the whole recording."""
    sh = es.shard
    S, K, T, dev = es.S, es.K, es.T, es.dev
    K2, tol = 2 * K, es.seam_tol
    lo = es.f_lo                  # first seam to check: 0 when a left neighbour rank sends chain 0's truth
    plan = es.plan
    plan.halo = plan.halo_next = int(es.halo)
    ops.set_chain_halos(plan)
    ll = es.emission(tuning)
    ops.phase("emission")
    bp = ops.viterbi_bp(T, K, dev)
    # message at the last bin of each chain, one slot ahead: seam c (in front of chain c) finds its truth in slot c;
    # slot 0 holds the left neighbour rank's last message
    end_ext = torch.zeros((S + 1, 2, K), dtype=torch.float32, device=dev)
    warm0 = getattr(es.op, "stationary", None)
    tail = es.tail
    tail.zero_()
    xbuf = torch.zeros(8 * K, dtype=torch.float32, device=dev) if sh.active else None

    def fwd(mode=0, ids=None, **sel):
        ops.viterbi_forward(plan, es.op, ll, bp, es.lmr, halo_state=(es.halo_state if mode == 0 else None),
                            end_msg=end_ext[1:], carry_in=es.carry_in, mode=mode, chain_ids=ids,
                            warm_in=(warm0 if mode == 0 else es.halo_state), **sel)

    def check(fix, slot, err, first=lo):
        if S > first:
            ops.seam_check_fix(S - first, K2, es.halo_state[first].data_ptr(), K2, end_ext[first].data_ptr(), K2,
                               err[first:S], tol, fix, tail[slot:slot + 1])

    def exchange():
        """last message to the right neighbour: the seam truth of its chain 0 (the filter's forward exchange)"""
        ops.boundary_pack_fwd(K, xbuf, None, end_ext[S])
        g = sh.neighbour_gather(xbuf)
        ops.boundary_unpack_fwd(K, None if sh.is_first else g[sh.rank - 1, 4 * K:], None, end_ext[0], None)

    def verdict():
        es._verdict_enqueue()                 # time-sharded: the record is summed over ranks
        err, fail, _ = es._verdict_wait()
        return err, fail

    fwd()
    if S > 1 and es.device_repair:
        check(True, T_FIX_F, es.err1, first=1)
        fwd(mode=2, sel_err=es.err1[:S], sel_tol=tol)
    if sh.active:
        ops.phase("viterbi_forward")
        exchange()
        ops.phase("exchange")
    check(False, T_FAIL_F, es.err)
    ops.phase("viterbi_forward")
    err, fail = verdict()
    n_fix, n_relay, n_relay_boundary = int(es.tail_host[T_FIX_F]), 0, 0
    # host (Jacobi) sweeps: the verdict is global, so every rank runs the same number of them
    for _ in range(es.max_sweeps):
        if not fail:
            break
        bad = torch.nonzero(~(err[lo:S] <= tol)).flatten() + lo
        n_relay += int(bad.numel())
        n_relay_boundary += int(lo == 0 and bool((bad == 0).any()))
        if bad.numel():
            idl = bad.to(dev)
            es.halo_state[idl] = end_ext[idl]                 # restart from the neighbour's current message
            fwd(mode=1, ids=idl.to(torch.int32))
        if sh.active:
            exchange()                # a restarted last chain changes the message the right neighbour checks against
        tail.zero_()
        check(False, T_FAIL_F, es.err)
        err, fail = verdict()
    if fail:
        raise SeamError("Viterbi: seams still above seam_tol=%g after %d repair sweeps (worst %.3g)"
                        % (tol, es.max_sweeps, float(err[lo:S].max()) if S > lo else float("nan")))
    if sh.active:
        ops.phase("viterbi_forward")
    maps = torch.empty((S, K2), dtype=torch.int32, device=dev)
    path = torch.empty(T, dtype=torch.int32, device=dev)
    ops.viterbi_chain_maps(plan, K, bp, maps)
    ops.phase("chain_maps")
    res = ViterbiResult()
    if sh.active:
        rec = ops.viterbi_records(1, K, dev)
        link, msg, lsum = ops.split_viterbi_records(rec, K)
        if not sh.is_first:
            ops.viterbi_block_link(plan, K, bp, maps, link[0])
        ops.phase("block_link")
        msg[0].copy_(end_ext[S].view(-1))
        lsum.copy_(es.lmr[es.core].sum(dtype=torch.float64))
        g = sh.neighbour_gather(rec.view(-1))                 # [world, 4K + 2]: the ONE exchange of the backtrack
        ops.phase("all_gather")
        ops.viterbi_backtrack_sharded(plan, K, bp, maps, g, sh.rank, path)
        ops.phase("backtrack")
        _, msgs, lsums = ops.split_viterbi_records(g, K)
        # the same gathered bytes on every rank -> the same value, bit for bit; partial sums added in rank order
        tot = 0.0
        for v in lsums.tolist():
            tot += v
        res.log_joint_map = torch.tensor(tot + float(torch.log(msgs[-1].max().double())), dtype=torch.float64)
    else:
        ops.viterbi_backtrack(plan, K, bp, maps, end_ext[S], path)
        ops.phase("backtrack")
        res.log_joint_map = es.lmr[es.core].sum(dtype=torch.float64) + torch.log(end_ext[S].max().double())
    res.path = path[es.core]
    res.n_fix, res.n_relay, res.n_relay_boundary, res.n_chain = n_fix, n_relay, n_relay_boundary, S
    res.seam_err = float(err[lo:S].max()) if S > lo else 0.0
    return res
