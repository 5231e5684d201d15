"""Time-sharded Viterbi decoding (decode_latent_viterbi(time_sharded=True)) at the headline shape N=500, K=400,
T=10^6, strong scaling: run with ``torchrun --nproc-per-node W scripts/bench_viterbi_sharded.py``.  Each rank holds
T/W bins.

Per rank, CUDA-event times (median of REPS) of the phases of one sharded decode: emission, the Viterbi forward pass
(seam checks, device repairs and host sweeps included), the boundary exchange after the pass, the chain maps,
pmg_viterbi_block_link, the all-gather of the backtrack records and pmg_viterbi_backtrack_sharded; and the end-to-end
decode_latent_viterbi(time_sharded=True).  In the same run rank 0 times the single-GPU decode of the whole recording
(its backtrack phase is what block_link is to be compared with) and checks that the concatenated sharded path equals
it.  With one GPU per rank the ranks talk over NCCL; on a box with fewer GPUs than ranks they share cuda:0 over gloo,
and only correctness is reported ("scaling_measured": false).  Prints one JSON line per measurement (rank 0)."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import torch.distributed as dist

import poor_man_gplvm_b200 as pmg
from poor_man_gplvm_b200 import ops, viterbi
from poor_man_gplvm_b200.estep import EStep
from poor_man_gplvm_b200.shard import TimeShard
from poor_man_gplvm_b200.synthetic import make_dataset_torch

REPS = 5
N, K, T = 500, 400, 1_000_000


def card(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(dev.index)],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                   # the number is reported without it, and says so
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


class Phases:
    """ops.PHASE_HOOK: a CUDA event per mark; the time since the previous mark is added to the mark's name."""

    def __init__(self):
        self.marks = []

    def __call__(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.marks.append((name, e))

    def totals(self):
        torch.cuda.synchronize()
        out = {}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out


def phase_medians(es, tun):
    viterbi.run(es, tun)                                     # warm-up
    runs, res = [], None
    for _ in range(REPS):
        ph = Phases()
        ops.PHASE_HOOK = ph
        ph("start")
        res = viterbi.run(es, tun)
        ops.PHASE_HOOK = None
        runs.append(ph.totals())
    return {k: round(float(np.median([r[k] for r in runs])), 4) for k in runs[0]}, res


def timed(fn, barrier=None):
    ts, out = [], None
    fn()
    for _ in range(REPS):
        if barrier:
            barrier()
        torch.cuda.synchronize()
        w0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - w0) * 1e3)
    return round(float(np.median(ts)), 3), [round(t, 3) for t in ts], out


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    nccl = torch.cuda.device_count() >= world
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)) if nccl else 0)
    torch.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist.init_process_group("gloo")
    name, pl = card(dev)
    d = make_dataset_torch(T, N, K, dev, seed=0)             # the same recording on every rank; each keeps its block
    y, tun = d["y"], d["tuning_true"].contiguous()
    lo, hi = rank * T // world, (rank + 1) * T // world
    y_blk = y[lo:hi].contiguous()
    if rank != 0:
        del y, d
    model = pmg.PoissonGPLVMJump1D(N, K, device=dev)
    P, logP, M, logM, op = model._transition_pack({})
    ma_n, ma_l = model._masks(None, None, hi - lo)
    es = EStep(y_blk, op, ma_n, ma_l, 1.0, shard=TimeShard())
    ph, res = phase_medians(es, tun)
    del es
    e2e, e2e_all, out = timed(lambda: model.decode_latent_viterbi(y_blk, tuning=tun, time_sharded=True,
                                                                  return_device=True), barrier=dist.barrier)
    mine = dict(rank=rank, n_chain=res.n_chain, seams_fixed_on_device=res.n_fix, seams_relayed_on_host=res.n_relay,
                rank_boundary_relays=res.n_relay_boundary, phases_ms=ph, end_to_end_ms=e2e, end_to_end_all=e2e_all,
                log_joint_map=out["log_joint_map"])
    flat = (out["map_dynamics"] * K + out["map_latent"]).cpu().numpy()
    per_rank = [None] * world
    paths = [None] * world
    dist.all_gather_object(per_rank, mine)
    dist.all_gather_object(paths, flat)
    if rank == 0:
        es1 = EStep(y, op, *model._masks(None, None, T), 1.0)
        ph1, res1 = phase_medians(es1, tun)
        del es1
        t1, t1_all, one = timed(lambda: model.decode_latent_viterbi(y, tuning=tun, return_device=True))
        same = bool(np.array_equal(np.concatenate(paths),
                                   (one["map_dynamics"] * K + one["map_latent"]).cpu().numpy()))
        lj_rel = abs(mine["log_joint_map"] - one["log_joint_map"]) / abs(one["log_joint_map"])
        common = dict(gpu=name, power_limit=pl, N=N, K=K, T=T, world=world, backend="nccl" if nccl else "gloo",
                      scaling_measured=nccl)
        if not nccl:
            common["note"] = "fewer GPUs than ranks: the ranks share cuda:0, scaling is not measured"
        print(json.dumps(dict(common, what="correctness", path_equal_to_single_gpu=same,
                              log_joint_map_rel_diff=lj_rel,
                              log_joint_map_identical_on_ranks=len({p["log_joint_map"] for p in per_rank}) == 1)),
              flush=True)
        for p in per_rank:
            print(json.dumps(dict(common, what="sharded_rank", **p)), flush=True)
        print(json.dumps(dict(common, what="single_gpu", phases_ms=ph1, end_to_end_ms=t1, end_to_end_all=t1_all,
                              n_chain=res1.n_chain)), flush=True)
        bl = max(p["phases_ms"].get("block_link", 0.0) for p in per_rank)
        print(json.dumps(dict(common, what="block_link_vs_single_gpu_backtrack", block_link_ms_max_over_ranks=bl,
                              single_gpu_backtrack_ms=ph1["backtrack"])), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
