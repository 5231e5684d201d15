"""Host-side orchestration of time-sharded Viterbi decoding (`viterbi.run` on a time-sharded `EStep`) on CPU: the
rank-boundary exchange, host repair sweeps in lockstep over the ranks, the record all-gather and the cross-rank
resolve, under gloo with 3 ranks against a single-process run and the fp64 oracle.

The CUDA operators are replaced by NumPy stand-ins with the same conventions (tests/cpu_viterbi_emulation.py and
tests/cpu_scan_emulation.py); `viterbi.run`, `EStep`, `TimeShard` and the plan are the product code.
"""
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

T_TOTAL, N, K, HALO, CHUNK, SEED = 1500, 12, 16, 4, 24, 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _patch():
    """Route the operators viterbi.run and EStep use to the CPU stand-ins; no CUDA call is left on their path."""
    os.environ["PMG_SCAN_COMPACT"] = "0"
    import cpu_scan_emulation as emu
    import cpu_viterbi_emulation as vemu
    from poor_man_gplvm_b200 import ops

    class _Props:
        multi_processor_count = 2

    class _Stream:
        def synchronize(self):
            pass

    torch.cuda.get_device_properties = lambda dev=None: _Props()
    torch.cuda.current_stream = lambda dev=None: _Stream()
    torch.Tensor.pin_memory = lambda self, *a, **k: self
    ops.seam_check_fix = emu.seam_check_fix
    ops.boundary_pack_fwd, ops.boundary_unpack_fwd = emu.boundary_pack_fwd, emu.boundary_unpack_fwd
    ops.EmissionOperands = emu.FakeEmission
    ops.scan_compact_supported = lambda op, scale: False
    for name in ("viterbi_forward", "viterbi_chain_maps", "viterbi_block_link", "viterbi_backtrack",
                 "viterbi_backtrack_sharded"):
        setattr(ops, name, getattr(vemu, name))


def _problem():
    from poor_man_gplvm_b200 import gp_kernel as gpk
    from poor_man_gplvm_b200.synthetic import make_dataset
    d = make_dataset(T_TOTAL, N, K, seed=SEED)
    P, logP, M, logM = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), 1.0, 0.02, 0.05)
    host = gpk.move_operator_host(K, 1.0, None, p_move_to_jump=0.02)
    return d, P, M, host


def _decode(rank, world):
    _patch()
    from poor_man_gplvm_b200 import ops, viterbi
    from poor_man_gplvm_b200.estep import EStep
    from poor_man_gplvm_b200.shard import TimeShard
    d, P, M, host = _problem()
    bounds = [0, 300, 1100, T_TOTAL] if world == 3 else [0, T_TOTAL]
    lo, hi = bounds[rank], bounds[rank + 1]
    y = torch.from_numpy(d["y"][lo:hi].copy())
    op = ops.MoveOperator(host, M, torch.device("cpu"), P0=P[0])
    es = EStep(y, op, None, None, 1.0, halo=HALO, chunk_len=CHUNK, shard=TimeShard() if world > 1 else None)
    res = viterbi.run(es, torch.from_numpy(d["tuning_true"].astype(np.float32)))
    return {"path": res.path.numpy().astype(np.int64), "lj": float(res.log_joint_map), "n_fix": res.n_fix,
            "n_relay": res.n_relay, "boundary": res.n_relay_boundary, "ll": es.ll[es.core].numpy().copy()}


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        q.put((rank, _decode(rank, world)))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _run(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    for r in range(world):
        assert isinstance(out[r], dict), out[r]
    return [out[r] for r in range(world)]


@pytest.fixture(scope="module")
def single():
    ctx = mp.get_context("spawn")          # the operator patches stay out of this process
    q = ctx.Queue()
    p = ctx.Process(target=_single_worker, args=(q,))
    p.start()
    out = q.get(timeout=600)
    p.join(timeout=60)
    assert isinstance(out, dict), out
    return out


def _single_worker(q):
    try:
        q.put(_decode(0, 1))
    except Exception:  # pragma: no cover
        import traceback
        q.put(traceback.format_exc())


def test_sharded_resolve_and_sweep_lockstep_match_single_process(single):
    from oracle import viterbi_ref as vr
    from poor_man_gplvm_b200 import gp_kernel as gpk
    outs = _run(3)
    path = np.concatenate([o["path"] for o in outs])
    np.testing.assert_array_equal(path, single["path"])
    assert len({o["lj"] for o in outs}) == 1                        # global, identical on every rank
    assert abs(outs[0]["lj"] - single["lj"]) <= 1e-6 * abs(single["lj"])
    # the 4-bin warm-ups miss seam_tol: interior seams are fixed "on the device", rank-boundary seams by host sweeps
    assert outs[0]["boundary"] == 0 and sum(o["boundary"] for o in outs[1:]) >= 1
    assert outs[0]["n_fix"] > 0
    # and the path is the MAP path of the oracle
    _, logP, _, logM = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), 1.0, 0.02, 0.05)
    ll = np.concatenate([o["ll"] for o in outs])
    opath, olj = vr.viterbi(ll, logP, logM)
    np.testing.assert_array_equal(path, opath)
    assert abs(outs[0]["lj"] - olj) <= 1e-6 * abs(olj)
