"""Shuffle significance test (poor_man_gplvm_b200.test.shuffle_test) on one GPU: end-to-end time of 100 circular
shuffles, per-phase device times (shifted prepare, emission, log-sum-exp / forward filter, quantile) and the
bandwidth of the shifted prepare on its compulsory bytes, for both decoders at the headline shape (N=500, K=400,
T=10^6) and a recording-sized one (N=200, K=100, T=2*10^5).  Baseline: shuffle_and_decode(keys=(sig_key,)) on a few
shuffles at the recording-sized shape (the full-key test_one_model cannot hold its results at the headline shape and
is not timed).  Device-generated data, one warm-up call, CUDA events.  Prints one JSON line per measurement."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import poor_man_gplvm_b200 as pmg
from poor_man_gplvm_b200 import batched, ops
from poor_man_gplvm_b200 import test as shuf
from poor_man_gplvm_b200.synthetic import make_dataset_torch

HBM_GBS = 6548.8        # sustained HBM bandwidth of one B200 used throughout DESIGN.md section 4
N_SHUFFLE = 100
SHAPES = [("headline", 500, 400, 1_000_000), ("recording", 200, 100, 200_000)]


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
        out = {}
        for (_, a), (name, b) in zip(self.marks, self.marks[1:]):
            out[name] = out.get(name, 0.0) + a.elapsed_time(b)
        return out


def timed(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record()
    r = fn()
    e1.record()
    torch.cuda.synchronize()
    return r, e0.elapsed_time(e1), (time.perf_counter() - w0) * 1e3


def run_shape(tag, N, K, T, name, pl):
    dev = torch.device("cuda", 0)
    d = make_dataset_torch(T, N, K, dev, seed=1)
    y = d["y"].to(torch.float32).contiguous()
    m = pmg.PoissonGPLVMJump1D(N, K, tuning_lengthscale=8.0)
    m.tuning = d["tuning_true"].to(torch.float32).contiguous()
    shifts = shuf.draw_shifts(T, N, N_SHUFFLE, seed=3)
    ld16 = (N + 7) // 8 * 8
    res = {}
    for dec in ("naive_bayes", "dynamics"):
        shuf.shuffle_test(m, y, n_shuffle=2, shifts=shifts[:2], decoder_type=dec)           # warm-up
        out, ev_ms, wall_ms = timed(lambda: shuf.shuffle_test(m, y, n_shuffle=N_SHUFFLE, shifts=shifts,
                                                              decoder_type=dec, return_device=True))
        # phase breakdown: the same steps through the session, every phase bracketed by events
        ses, setup_ms, _ = timed(lambda: batched.DecodeSession(m, y))
        ph = Phases()
        ops.PHASE_HOOK = ph
        try:
            ph("start")
            rows = ses.shuffled(shifts, dec)
            batched.quantile_rows(rows, 0.975)
            ph("quantile")
        finally:
            ops.PHASE_HOOK = None
        t = ph.totals()
        prep_bytes = N_SHUFFLE * T * (2 * N + 2 * (ld16 if dec == "naive_bayes" else (N + 8) // 8 * 8) + 4)
        gbs = prep_bytes / (t["shifted_prepare"] * 1e-3) / 1e9
        line = {"shape": tag, "N": N, "K": K, "T": T, "decoder": dec, "n_shuffle": N_SHUFFLE,
                "shuffle_test_ms": round(ev_ms, 2), "shuffle_test_wall_ms": round(wall_ms, 2),
                "ms_per_shuffle": round(ev_ms / N_SHUFFLE, 3), "session_setup_ms": round(setup_ms, 2),
                "phases_ms": {k: round(v, 3) for k, v in t.items()},
                "shifted_prepare_GBps": round(gbs, 1), "shifted_prepare_frac_of_6548.8": round(gbs / HBM_GBS, 3),
                "shifted_prepare_bytes": prep_bytes, "n_sig": int(out["is_sig_tsd"].sum().item()),
                "gpu": name, "power_limit": pl}
        print(json.dumps(line), flush=True)
        res[dec] = (out, shifts)
        del ses, rows, out
        torch.cuda.empty_cache()
    return m, y, res


def baseline(m, y, res, name, pl, n_base=3):
    for dec, key in batched.SIG_KEYS.items():
        out, shifts = res[dec]
        shuf.shuffle_and_decode(m, y, n_shuffle=1, decoder_type=dec, shifts=shifts, keys=(key,))      # warm-up
        r, ev_ms, wall_ms = timed(lambda: shuf.shuffle_and_decode(m, y, n_shuffle=n_base, decoder_type=dec,
                                                                  shifts=shifts, keys=(key,)))
        got = out["sig_shuffle"][:n_base].cpu().numpy()
        diff = float(np.max(np.abs(got - r[key])))
        print(json.dumps({"baseline": "shuffle_and_decode(keys=(sig_key,))", "shape": "recording", "decoder": dec,
                          "n_shuffle": n_base, "ms_per_shuffle": round(ev_ms / n_base, 2),
                          "wall_ms_per_shuffle": round(wall_ms / n_base, 2),
                          "max_abs_diff_vs_shuffle_test": diff, "gpu": name, "power_limit": pl}), flush=True)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("bench_shuffle_test.py needs a CUDA device")
    torch.cuda.set_device(0)
    name, pl = card()
    print(json.dumps({"gpu": name, "power_limit": pl,
                      "note": "test_one_model (all result keys) is not timed at the headline shape: "
                              "it stacks every key of every shuffle on the host (~480 GB for naive Bayes)"}),
          flush=True)
    for tag, N, K, T in SHAPES:
        m, y, res = run_shape(tag, N, K, T, name, pl)
        if tag == "recording":
            baseline(m, y, res, name, pl)
        del m, y, res
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
