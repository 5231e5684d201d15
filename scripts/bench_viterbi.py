"""Viterbi decoding (decode_latent_viterbi) on one GPU at the headline shape N=500, K=400, T=10^6: CUDA-event times of
the emission GEMM, the Viterbi forward pass (seam checks and device repairs included), the chain maps and the
backtrack, with the achieved bandwidth of the two scans on their algorithmic bytes:

  forward: ll read (4K B/bin) + backpointers written (2K int16 = 4K B/bin);  chain maps: backpointers read once.

decode_latent and decode_latent_viterbi are timed end to end in the same run.  Device-generated data (the planted
tuning), one warm-up call per measurement, median of REPS repetitions.  Prints one JSON line per measurement."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import poor_man_gplvm_b200 as pmg
from poor_man_gplvm_b200 import ops, viterbi
from poor_man_gplvm_b200.estep import EStep
from poor_man_gplvm_b200.synthetic import make_dataset_torch

HBM_GBS = 6548.8        # sustained HBM bandwidth of one B200 used throughout DESIGN.md section 4
REPS = 5
N, K, T = 500, 400, 1_000_000


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                   # the number is reported without it, and says so
        pl = "unknown (%s)" % type(e).__name__
    return name, pl


class Phases:
    """ops.PHASE_HOOK: a CUDA event per mark; the time since the previous mark goes to the mark's name."""

    def __init__(self):
        self.marks = []

    def __call__(self, name):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        self.marks.append((name, e))

    def totals(self):
        torch.cuda.synchronize()
        return {name: a.elapsed_time(b) for (_, a), (name, b) in zip(self.marks, self.marks[1:])}


def timed(fn):
    torch.cuda.synchronize()
    w0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - w0) * 1e3, out


def main():
    torch.cuda.set_device(0)
    name, pl = card()
    dev = torch.device("cuda", 0)
    d = make_dataset_torch(T, N, K, dev, seed=0)
    y, tun = d["y"].contiguous(), d["tuning_true"].contiguous()
    model = pmg.PoissonGPLVMJump1D(N, K, device=dev)
    P, logP, M, logM, op = model._transition_pack({})
    ma_n, ma_l = model._masks(None, None, T)
    es = EStep(y, op, ma_n, ma_l, 1.0)
    viterbi.run(es, tun)                                     # warm-up
    phases, res = [], None
    for _ in range(REPS):
        ph = Phases()
        ops.PHASE_HOOK = ph
        ph("start")
        res = viterbi.run(es, tun)
        ops.PHASE_HOOK = None
        phases.append(ph.totals())
    med = {k: float(np.median([p[k] for p in phases])) for k in phases[0]}
    bytes_fwd = T * (4 * K + 2 * 2 * K)
    bytes_maps = T * 2 * 2 * K
    common = dict(gpu=name, power_limit=pl, N=N, K=K, T=T, n_chain=res.n_chain, seams_fixed_on_device=res.n_fix,
                  seams_relayed_on_host=res.n_relay)
    print(json.dumps(dict(common, what="viterbi_phases_ms", **{k: round(v, 4) for k, v in med.items()},
                          forward_GBps=round(bytes_fwd / med["viterbi_forward"] / 1e6, 1),
                          forward_share_of_hbm=round(bytes_fwd / med["viterbi_forward"] / 1e6 / HBM_GBS, 3),
                          maps_GBps=round(bytes_maps / med["chain_maps"] / 1e6, 1),
                          maps_share_of_hbm=round(bytes_maps / med["chain_maps"] / 1e6 / HBM_GBS, 3))),
          flush=True)
    for what, fn in (("decode_latent_viterbi_ms", lambda: model.decode_latent_viterbi(y, tuning=tun,
                                                                                      return_device=True)),
                     ("decode_latent_ms", lambda: model.decode_latent(y, tuning=tun, return_device=True))):
        fn()
        ts = [timed(fn)[0] for _ in range(REPS)]
        print(json.dumps(dict(common, what=what, median=round(float(np.median(ts)), 3),
                              all=[round(t, 3) for t in ts])), flush=True)


if __name__ == "__main__":
    main()
