#!/usr/bin/env python
"""bench.py — EM throughput of the PoissonGPLVMJump1D hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this framework
  python bench.py --impl reference --steps K --warmup W    # restated reference on the host CPU

A "step" is ONE EM iteration (sufficient statistics -> Adam M-step -> emission ->
forward -> backward) over the whole synthetic spike matrix of the workload
(default: BASELINE.json configs[3], N=500 neurons, K=400 latent bins, T=1e6 bins).
`value` = T * steps / device time with the spikes resident in HBM;
`e2e`   = T * n_iter / wall time of a full `fit_em` call on HOST arrays (H2D of the
          spikes and D2H of every result array inside the timed region; median of 3 calls).
With --gpus N the recording is time-sharded over N ranks.  --scaling strong (default,
BASELINE.json's north star): ONE recording of T bins split over the ranks; --scaling weak:
every rank holds T bins of an N*T-bin recording.  In strong mode rank 0 also fits the first
iterations of the same recording alone and the line carries `parity_vs_1rank`.
--workload nb is configs[2] (decode_latent_naive_bayes only; metric: decode bins/s).
--dump-outputs DIR writes what the last timed step computed to DIR/<name>.npy (rank 0; the inputs are seeded, so
two builds run with the same arguments can be compared array for array).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N, K, T, tuning_lengthscale, movement_variance)
    "readme": (30, 100, 1000, 10.0, 1.0),
    "session": (200, 100, 100000, 10.0, 1.0),
    "headline": (500, 400, 1000000, 10.0, 1.0),
    "stress": (300, 2000, 1000000, 10.0, 1.0),          # K = 2000 with the default (11-tap) move kernel
    # BASELINE configs[4] as written: a DENSE K x K move kernel (custom_transition_kernel, gp_kernel.py:61-66)
    # dominating the scan -> the lockstep tensor-core scan (pmg_forward_dense / pmg_backward_dense)
    "stress_dense": (300, 2000, 1000000, 10.0, 1.0),
    "nb": (1000, 200, 10000000, 10.0, 1.0),
}
METRIC = "EM time-bins x iters/s"
UNIT = "bins*iters/s"
NB_METRIC = "decode bins/s (decode_latent_naive_bayes)"
NCU_SUMMARY = "profiles/r02_ncu_full_summary.csv"
DUMP_LIMIT = 64 * 10 ** 6          # bytes written by --dump-outputs in all
DUMP_TIME_BUDGET = 48 * 10 ** 6    # of which the T-sized arrays (row sample); the rest: tuning, weights, histories


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


def ncu_traffic():
    """DRAM bytes per launch of the hot kernels from the committed ncu --set full summary (headline workload)."""
    path = os.path.join(ROOT, NCU_SUMMARY)
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r01_ncu_full_summary_v4.csv")
    out = {}
    try:
        import csv
        with open(path) as f:
            for rec in csv.DictReader(f):
                def gb(x):
                    v, u = x.split()
                    return float(v) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[u]
                full = rec["kernel"].replace("void ", "").split("(")[0]
                name = full.split("<")[0]
                val = gb(rec["dram__bytes_read.sum"]) + gb(rec["dram__bytes_write.sum"])
                out[full.replace(" ", "")] = val              # e.g. atb_tc_kernel<1,0> (statistics) vs <2,1> (xi)
                out.setdefault(name, val)
    except Exception:
        return {}
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    PERIOD_MS = 20

    def __init__(self, index=0):
        self.index, self.proc = index, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", str(self.PERIOD_MS)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self, t_begin=None, t_end=None):
        """Samples whose nvidia-smi timestamp falls inside [t_begin, t_end] (time.time() values) -- the sampler
        is started well before the timed region because nvidia-smi needs ~0.2 s to produce its first line."""
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        import datetime
        sm, mx, reasons, n_all = [], [], set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            n_all += 1
            if t_begin is not None:
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                except ValueError:
                    continue
                if ts < t_begin - 0.02 or ts > t_end + 0.02:
                    continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "samples_outside_timed_region": n_all - len(sm), "reasons": sorted(reasons)}


def dump_rows(T, row_bytes):
    """Time bins kept by --dump-outputs: all of them when the T-sized arrays fit DUMP_TIME_BUDGET, otherwise a
    sorted draw without replacement from a fixed seed (the same bins for every build at the same T)."""
    n = DUMP_TIME_BUDGET // max(1, row_bytes)
    if T <= n:
        return np.arange(T)
    return np.sort(np.random.default_rng(0).choice(T, size=n, replace=False))


def write_dump(out_dir, arrays):
    """name -> tensor / array / scalar, written as out_dir/<name>.npy; float32 stays float32, everything else is
    stored as float64 (exact for the iteration counts and bin indices)."""
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        host[name] = a if a.dtype == np.float32 else a.astype(np.float64)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# reference arm: the restated reference (oracle/ref_numpy.py, fp32, reference operation order) on the host
# ------------------------------------------------------------------------------------------------
def cpu_reference_rate(N, K, ls, mv, sample_T, n_steps, n_warm, full_T, seed=0):
    """Times EM iterations of the NumPy restatement on a bounded sample of the workload: `sample_T` bins of the
    same synthetic process, walked as TWO reference chunks (n_time_per_chunk = sample_T / 2, so the chunk loop of
    decoder.py:283-324 with its carried messages is on the timed path).  The E-step and the statistics GEMM cost
    is linear in T; the Adam M-step is T-independent.  BLAS is pinned to one thread (the restatement's time goes
    into single-threaded NumPy transcendentals either way), so `cores` = 1 is what was used.  Returns the rate
    extrapolated to the full workload, T / (t_mstep + (T / sample_T) * t_estep_and_stats), and the measured parts."""
    from threadpoolctl import threadpool_limits
    from oracle import ref_numpy as ref
    from poor_man_gplvm_b200.synthetic import make_dataset
    from poor_man_gplvm_b200 import gp_kernel as gpk

    d = make_dataset(sample_T, N, K, seed=seed)
    basis = gpk.generate_basis(ls, K)
    rng = np.random.default_rng(seed + 1)
    params = rng.standard_normal((basis.shape[1], N)).astype(np.float32)
    m = ref.OraclePoissonGPLVMJump1D(N, K, tuning_lengthscale=ls, movement_variance=mv, dtype=np.float32,
                                     tuning_basis=basis, params=params)
    y = d["y"].astype(np.float32)
    _, logP, _, logM = m._transitions({})
    with np.errstate(over="ignore"):
        lp, _ = m.init_latent_posterior(sample_T, seed)
    opt = ref.adam_init(m.params)
    W = m.params
    chunk = max(1, (sample_T + 1) // 2)
    t_m, t_e = [], []
    with threadpool_limits(limits=1):
        for it in range(n_warm + n_steps):
            t0 = time.perf_counter()
            yw, tw = ref.get_statistics(lp, y)
            t1 = time.perf_counter()
            res = ref.adam_run(W, opt, 1.0, basis, yw, tw, step_size=0.01, maxiter=1000, tol=1e-6)
            W, opt = res["params"], res["opt_state"]
            tuning = ref.get_tuning_softplus(W, basis)
            t2 = time.perf_counter()
            out = ref.smooth_all_step_combined_ma_chunk(y, tuning, logP, logM, m.ma_neuron_default,
                                                        m.ma_latent_default, 1.0, chunk, accumulate=True)
            lp = ref.lse(out[0], axis=1)
            t3 = time.perf_counter()
            if it >= n_warm:
                t_m.append(t2 - t1)
                t_e.append((t1 - t0) + (t3 - t2))
    tm, te = float(np.mean(t_m)), float(np.mean(t_e))
    sec_full = tm + te * (full_T / sample_T)
    return full_T / sec_full, {"t_mstep_s": tm, "t_estep_sample_s": te, "sample_bins": sample_T, "chunk_bins": chunk,
                               "sec_per_iter_extrapolated": sec_full}


def cpu_nb_rate(N, K, sample_T, seed=0):
    """decode_latent_naive_bayes of the NumPy restatement (decoder.py:88-149, two chunks) on `sample_T` bins."""
    from threadpoolctl import threadpool_limits
    from oracle import ref_numpy as ref
    from poor_man_gplvm_b200.synthetic import make_dataset
    d = make_dataset(sample_T, N, K, seed=seed)
    tun = d["tuning_true"].astype(np.float32)
    with threadpool_limits(limits=1):
        t0 = time.perf_counter()
        ref.get_naive_bayes_ma_chunk(d["y"].astype(np.float32), tun, np.ones(N, np.float32), np.ones(K, np.float32),
                                     1.0, max(1, (sample_T + 1) // 2))
        sec = time.perf_counter() - t0
    return sample_T / sec, sec


def reference_sample_bins(args, rate_guess=110.0):
    """bins per step of the reference arm: the whole `--steps K --warmup W` run should end within ~3 minutes
    (measured: ~110 bins/s for the log-space E-step at N=500, K=400), never less than two chunks of 100 bins."""
    if args.cpu_sample_bins:
        return args.cpu_sample_bins
    budget = 170.0 / max(1, args.steps + args.warmup)
    return int(min(2000, max(200, rate_guess * budget)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, K, T, ls, mv = WORKLOADS[args.workload]
    if args.workload == "nb":
        sample_T = args.cpu_sample_bins or 400
        for _ in range(args.warmup):
            cpu_nb_rate(N, K, sample_T)
        rates = [cpu_nb_rate(N, K, sample_T)[0] for _ in range(args.steps)]
        rate = float(np.median(rates))
        line = {"impl": "reference", "metric": NB_METRIC, "value": rate, "unit": "bins/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": sample_T / rate * 1e3,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": "nb: N=%d K=%d T=%d (CPU arm timed on %d bins/step)" % (N, K, T, sample_T)},
                "cpu_baseline": {"value": rate, "unit": "bins/s", "cores": 1, "kind": "port",
                                 "sample": "%d bins per step, two reference chunks; restated reference (NumPy CPU, "
                                           "fp32), not JAX" % sample_T},
                "e2e": {"value": rate, "unit": "bins/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return
    sample_T = reference_sample_bins(args)
    rate, parts = cpu_reference_rate(N, K, ls, mv, sample_T, args.steps, args.warmup, T)
    sec = parts["t_mstep_s"] + parts["t_estep_sample_s"]
    sample = ("%d-bin sample of the workload per step, walked as two reference chunks of %d bins (one EM iteration: "
              "default Adam M-step %.2f s, T-independent; statistics + chunked log-space filter/smoother with the "
              "[2,2,K,K] joint accumulation %.2f s, linear in T); value = T/(t_mstep + T/%d * t_estep) extrapolated "
              "to T=%d" % (sample_T, parts["chunk_bins"], parts["t_mstep_s"], parts["t_estep_sample_s"], sample_T, T))
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "%s: N=%d K=%d T=%d (CPU arm timed on %d bins/step)" % (args.workload, N, K, T, sample_T)},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": sample + "; restated reference (NumPy CPU, BLAS pinned to 1 thread), not JAX: "
                                                "jax/optax are not installable here"},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# this framework
# ------------------------------------------------------------------------------------------------
class PhaseTimer:
    """CUDA events around each phase of an EM iteration (on the launching stream).  The launching thread
    synchronises at every mark, so each phase is timed alone: start event, the phase's launches, end event."""

    def __init__(self, torch):
        self.torch = torch
        self.spans = []
        self.n_begin = 0
        self.enabled = False
        self._start = None
        self._host0 = 0.0

    def hook(self, name):
        if not self.enabled:
            return
        host1 = time.perf_counter()
        if name == "begin":
            self.n_begin += 1
        elif self._start is not None:
            end = self.torch.cuda.Event(enable_timing=True)
            end.record()
            self.spans.append((name, self._start, end, (host1 - self._host0) * 1e3))
        self.torch.cuda.synchronize()
        self._start = self.torch.cuda.Event(enable_timing=True)
        self._start.record()
        self._host0 = time.perf_counter()

    def summarize(self):
        tot = {}
        for name, e0, e1, _ in self.spans:
            tot[name] = tot.get(name, 0.0) + e0.elapsed_time(e1)
        return tot

    def summarize_host(self):
        """Host-side time of the same spans (launch overhead of each phase, not GPU time)."""
        tot = {}
        for name, _, _, h in self.spans:
            tot[name] = tot.get(name, 0.0) + h
        return tot


def _setup_dist(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1:
        raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    one_gpu = os.environ.get("PMG_BENCH_BACKEND", "nccl") == "gloo"     # emulation: all ranks share cuda:0
    dev = torch.device("cuda", 0 if one_gpu else local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        if one_gpu:
            dist.init_process_group("gloo")
        else:
            dist.init_process_group("nccl", device_id=dev)
    return torch, dist, world, rank, dev


def _block(total, world, rank):
    lo = rank * total // world
    hi = (rank + 1) * total // world
    return lo, hi


def run_nb(args):
    """configs[2]: decode_latent_naive_bayes only (emission GEMM + row normalisation), time-sharded without any
    data-path collective; value = bins decoded by all ranks / max-over-ranks device time."""
    torch, dist, world, rank, dev = _setup_dist(args)
    import poor_man_gplvm_b200 as pmg
    from poor_man_gplvm_b200 import ops
    from poor_man_gplvm_b200.synthetic import make_dataset_torch
    N, K, T, ls, mv = WORKLOADS["nb"]
    if args.bins:
        T = args.bins
    lo, hi = _block(T, world, rank) if args.scaling == "strong" else (0, T)
    Tr = hi - lo
    data = make_dataset_torch(Tr, N, K, dev, seed=4321 + rank, tuning_seed=4321)
    y_dev = data["y"].to(torch.float32).contiguous()
    tun = (data["tuning_true"] * 1.05).contiguous()
    model = pmg.PoissonGPLVMJump1D(N, K, tuning_lengthscale=ls, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        model.decode_latent_naive_bayes(y_dev, tuning=tun, return_device=True)
    barrier()
    l0 = ops.LAUNCHES
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        out = model.decode_latent_naive_bayes(y_dev, tuning=tun, return_device=True)
    ev1.record()
    barrier()
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    launches = ops.LAUNCHES - l0
    if args.dump_outputs and rank == 0:
        # the decode of the last timed step (this rank's block); T-sized arrays on a fixed sample of bins
        rows = dump_rows(Tr, 4 * (3 * K + 1))
        idx = torch.from_numpy(rows).to(dev)
        dump = {k: (v.index_select(0, idx) if torch.is_tensor(v) else v) for k, v in out.items()}
        dump["bins"] = rows
        write_dump(args.dump_outputs, dump)
    del out
    # end to end: host spikes in, argmax decode + posterior out (the arrays a user reads), median of 3
    y_host = y_dev.cpu().numpy()
    walls = []
    for i in range(4):
        barrier()
        t0 = time.perf_counter()
        r = model.decode_latent_naive_bayes(y_host, tuning=tun)
        torch.cuda.synchronize()
        if i:
            walls.append(time.perf_counter() - t0)
        d2h = sum(int(v.nbytes) for v in r.values() if isinstance(v, np.ndarray))
        del r
    wall = float(np.median(walls))
    if world > 1:
        t = torch.tensor([ms, wall], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0]), float(t[1])
    total = T if args.scaling == "strong" else T * world
    pk = peaks()
    if rank == 0:
        sec = ms * 1e-3 / args.steps
        flops = 2.0 * Tr * N * K
        cpu_rate, cpu_sec = cpu_nb_rate(N, K, args.cpu_sample_bins or 400) if not args.no_cpu_baseline else (None, None)
        line = {"metric": NB_METRIC, "value": total / sec, "unit": "bins/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "nb: N=%d K=%d T=%d bins total, %d per rank" % (N, K, total, Tr),
                           "parallelism": "time-sharded x%d, no data-path collective" % world,
                           "l2": "inputs larger than L2"},
                "roofline": {"bound": "tensor", "achieved": flops / sec / 1e12, "peak": pk["bf16_tflops"] / 2.0,
                             "unit": "TFLOP/s", "frac": flops / sec / 1e12 / (pk["bf16_tflops"] / 2.0),
                             "traffic": None, "kernel": "emission_tc_kernel + nb_normalize_kernel (whole decode)",
                             "peak_source": pk["src"] + " bf16 burst / 2 (derived TF32 dense)"},
                "cpu_baseline": None if cpu_rate is None else
                {"value": cpu_rate, "unit": "bins/s", "cores": 1, "kind": "port",
                 "sample": "%d bins, two reference chunks, %.1f s; restated reference (NumPy CPU), not JAX"
                           % (args.cpu_sample_bins or 400, cpu_sec)},
                "e2e": {"value": total / wall, "unit": "bins/s", "h2d_bytes_per_step": int(y_host.nbytes),
                        "d2h_bytes_per_step": d2h, "wall_s": wall, "n_calls": len(walls)},
                "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_ours(args):
    if args.workload == "nb":
        return run_nb(args)
    torch, dist, world, rank, dev = _setup_dist(args)
    import poor_man_gplvm_b200 as pmg
    from poor_man_gplvm_b200 import ops
    from poor_man_gplvm_b200.core import EMLoop
    from poor_man_gplvm_b200.shard import TimeShard
    from poor_man_gplvm_b200.synthetic import make_dataset_torch

    N, K, T, ls, mv = WORKLOADS[args.workload]
    if args.bins:
        T = args.bins
    strong = args.scaling == "strong"
    mk = {}
    if args.workload == "stress_dense":
        xk = np.arange(K, dtype=np.float64)
        mk["custom_transition_kernel"] = (np.exp(-np.abs(xk[:, None] - xk[None, :]) / 150.0) + 0.02).astype(np.float32)
    model = pmg.PoissonGPLVMJump1D(N, K, tuning_lengthscale=ls, movement_variance=mv, device=dev, **mk)
    rng = np.random.default_rng(1)
    model.params = rng.standard_normal((model.n_basis, N)).astype(np.float32)
    P, logP, M, logM, op = model._transition_pack({})

    def draw_init(n, seed):
        g = torch.Generator(device=dev); g.manual_seed(seed)
        post0 = torch.rand((n, K), generator=g, device=dev)
        return torch.log(post0 / post0.sum(dim=1, keepdim=True))

    if strong:
        # ONE recording of T bins; rank r owns bins [r*T/world, (r+1)*T/world).  Every rank generates the same
        # recording (same seed) and keeps its block, so the sharded fit and a single-rank fit see identical data.
        y_full = make_dataset_torch(T, N, K, dev, seed=1234, tuning_seed=1234)["y"].to(torch.float32).contiguous()
        lp_full = draw_init(T, 99)
        lo, hi = _block(T, world, rank)
        y_dev, lp0 = y_full[lo:hi].contiguous(), lp_full[lo:hi].contiguous()
        if not (world > 1 and rank == 0 and not args.no_parity):
            del y_full, lp_full
            y_full = lp_full = None
        T_rank, T_total = hi - lo, T
    else:
        # weak scaling: every rank owns T bins of ONE recording of world*T bins (same neurons and tuning curves on
        # every rank; each block has its own latent trajectory, spikes and rows of the iid initial posterior)
        y_dev = make_dataset_torch(T, N, K, dev, seed=1234 + rank, tuning_seed=1234)["y"].to(torch.float32).contiguous()
        lp0 = draw_init(T, 99 + 7919 * rank)
        y_full = lp_full = None
        T_rank, T_total = T, T * world
    ma_n, ma_l = model._masks(None, None, T_rank)
    shard = TimeShard() if world > 1 else None

    def new_loop(y, lp, sh, maxiter=None, tol=None):
        return EMLoop(model, y, op, ma_n, ma_l, 1.0, model.tuning_basis, lp, model.param_prior_std, 0.01,
                      args.m_step_maxiter if maxiter is None else maxiter, args.m_step_tol if tol is None else tol,
                      shard=sh)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity of the sharded fit against a single-rank fit of the same recording (strong mode, world > 1):
    # first iterations from the same initial posterior; log marginal per iteration and the tuning after them.
    # The Adam step count is pinned (25 steps, tol < 0) as in the parity tests: with the default stopping rule the
    # step at which a relative loss change of 1e-6 is reached depends on rounding (summation order over ranks), and
    # a fit that stops a few steps earlier differs in the tuning by the optimiser's tolerance, not by the sharding.
    parity = None
    if world > 1 and strong and not args.no_parity:
        n_par = args.parity_iters
        lp_s = new_loop(y_dev, lp0, shard, maxiter=25, tol=-1.0)
        lml_s = []
        for _ in range(n_par):
            r_, m_ = lp_s.iteration(speculate=True)
            lml_s.append(float(r_.log_marginal))
        tun_s = m_[4].clone()
        del lp_s
        barrier()
        if rank == 0:
            ma_full = model._masks(None, None, T)
            one = EMLoop(model, y_full, op, ma_full[0], ma_full[1], 1.0, model.tuning_basis, lp_full,
                         model.param_prior_std, 0.01, 25, -1.0, shard=None)
            lml_1 = []
            for _ in range(n_par):
                r_, m_ = one.iteration(speculate=True)
                lml_1.append(float(r_.log_marginal))
            tun_1 = m_[4]
            a, b = np.array(lml_s), np.array(lml_1)
            parity = {"iters": n_par, "adam": "25 steps per iteration (pinned)", "log_marginal_rel": float(np.max(np.abs(a - b) / np.abs(b))),
                      "tuning_rel": float(((tun_s - tun_1).abs() / tun_1).max().item()),
                      "tol": {"log_marginal_rel": 1e-4, "tuning_rel": 1e-3}}
            parity["ok"] = bool(parity["log_marginal_rel"] < 1e-4 and parity["tuning_rel"] < 1e-3)
            del one, tun_1
        del y_full, lp_full, tun_s
        torch.cuda.empty_cache()
        barrier()

    loop = new_loop(y_dev, lp0, shard)
    del lp0

    timer = PhaseTimer(torch)
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        loop.iteration(speculate=True)
    barrier()
    launches0 = ops.LAUNCHES
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall_begin = time.time()
    ev0.record()
    relays = fixes = 0
    n_adam, halos = [], []
    for _ in range(args.steps):
        res, m_res = loop.iteration(speculate=True)      # as fit_em runs every iteration but its last
        relays += res.n_relay_fwd + res.n_relay_bwd
        fixes += res.n_fix_fwd + res.n_fix_bwd
        halos.append(res.halo)
        n_adam.append(m_res[2])
    ev1.record()
    barrier()
    wall_end = time.time()
    clocks = sampler.stop(wall_begin, wall_end) if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    launches = ops.LAUNCHES - launches0
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    # replicated M-step: the tuning must be bit-identical on every rank
    tuning_identical = None
    if world > 1:
        tu = m_res[4].clone()
        ref_t = tu.clone()
        shard.broadcast_(ref_t, 0)
        d = (tu != ref_t).sum().to(torch.float32).reshape(1)
        shard.allreduce_flat_sum_(d)
        tuning_identical = bool(d.item() == 0)
    if args.dump_outputs and rank == 0:
        # what the last timed iteration handed its caller: its M-step (tuning, the GLM weights behind it, the Adam
        # record) and its E-step (log marginal, latent posterior of this rank's block on a fixed sample of bins)
        n_it = int(m_res[2].item())
        rows = dump_rows(T_rank, 4 * K)
        idx = torch.from_numpy(rows).to(dev)
        if res.gamma_lat is not None:
            post = res.gamma_lat.index_select(0, idx)
        else:       # tensor-core statistics: the posterior is kept as fp16 hi/lo pieces (ops.new_gamma16)
            g = loop.gamma16[:, loop.es.core, :K].index_select(1, idx)
            post = g[0].float() + g[1].float()
        write_dump(args.dump_outputs, {
            "tuning": m_res[4], "params": loop.W_iter, "log_marginal": res.log_marginal,
            "m_step_n_iter": n_it, "m_step_final": m_res[3], "m_step_loss_history": m_res[0][:n_it],
            "m_step_error_history": m_res[1][:n_it], "posterior_latent_marg": post, "posterior_bins": rows})
    # Per-phase CUDA events are taken in a SECOND pass of the same number of EM iterations, outside the timed
    # region, with the launching thread synchronising at every mark (each phase timed alone).  Events inside the
    # free-running loop perturb it (an event recorded between the cooperative M-step launch and the next launch
    # stalls the launching thread on this driver), which would be charged to the headline number.
    n_phase = args.phase_steps if args.phase_steps is not None else args.steps
    if n_phase > 0:
        loop.iteration()             # consumes the M-step the last timed iteration enqueued ahead (not instrumented)
    # (the hook also keeps these iterations out of the CUDA graph: each phase is launched and timed by itself)
    ops.PHASE_HOOK = timer.hook
    timer.enabled = True
    for _ in range(n_phase):
        timer.hook("begin")
        loop.iteration()
    torch.cuda.synchronize()
    timer.enabled = False
    phases = timer.summarize()
    phases_host = {k: v / max(1, timer.n_begin) for k, v in timer.summarize_host().items()}
    n_adam = [int(x.item()) for x in n_adam]
    ops.PHASE_HOOK = None
    value = T_total * args.steps / (ms * 1e-3)

    # ---- roofline of the dominant kernel (algorithmic bytes / flops per launch; DESIGN.md section 4)
    pk = peaks()
    S = max(1, timer.n_begin)
    per = {k: v / S for k, v in phases.items()}     # ms per EM iteration per phase (second, instrumented pass)
    # Algorithmic amounts per launch (DESIGN.md section 4).  Scans: the compulsory HBM bytes of the kernel variant
    # that ran.  EM-mode (compact) kernels: forward reads ll (4K) and writes the compact filtered posterior
    # (4K+16 per bin); backward reads ll and that buffer and writes the fp16 hi/lo pieces of gamma_lat (4K):
    # 8K and 12K bytes per bin.  General kernels (and SURVEY.md section 8(d)'s reference layout): 12K and 20K
    # bytes per bin -- reported beside as "survey_bytes".  GEMMs: one fp32-equivalent GEMM, 2*T*N*K flop.
    compact = bool(loop.es.compact_ok and loop.use_tc)
    Tr = T_rank
    dense = getattr(op, "dense", None) is not None
    algo = {
        "forward": ("hbm", (8.0 * K + 16.0) * Tr if compact else 12.0 * K * Tr, 12.0 * K * Tr),
        "backward": ("hbm", 12.0 * K * Tr if compact else 16.0 * K * Tr, 20.0 * K * Tr),
        "emission": ("tensor", 2.0 * Tr * N * K, None),
        "stats": ("tensor", 2.0 * Tr * N * K, None),
    }
    kernel_of = {"forward": "fwd_c_kernel" if compact else "fwd_bulk_kernel",
                 "backward": "bwd_c_kernel" if compact else "bwd_bulk_kernel",
                 "emission": "emission_tc2_kernel", "stats": "atb_tc_kernel<1,0>"}
    if dense:
        # lockstep scan: one K x K mat-vec per bin and pass = 2 K^2 fp32-equivalent flop (the warm-up bins and the
        # three fp16-piece products that realise one fp32-grade product are overhead, not algorithmic work)
        algo["forward"] = algo["backward"] = ("tensor", 2.0 * K * K * Tr, None)
        kernel_of["forward"] = kernel_of["backward"] = "dense_step_gemm_kernel (+ dense_*_update_kernel)"
    traffic = ncu_traffic() if (args.workload == "headline" and not args.bins and world == 1) else {}
    roof_all = {}
    for name, (bound, amount, survey) in algo.items():
        if name not in per or per[name] <= 0:
            continue
        sec = per[name] * 1e-3
        if bound == "hbm":
            ach, peak, unit = amount / sec / 1e9, pk["hbm_gbs"], "GB/s"
        else:
            # fp32-equivalent GEMM flops against the derived TF32 dense peak = measured bf16 BURST / 2: every phase
            # of this pass is timed alone (synchronisation at each mark), i.e. a kernel timed by itself
            ach, peak, unit = amount / sec / 1e12, pk["bf16_tflops"] / 2.0, "TFLOP/s"
        roof_all[name] = {"bound": bound, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak,
                          "ms": per[name], "kernel": kernel_of[name], "algorithmic": amount,
                          "traffic": traffic.get(kernel_of[name])}
        if bound == "tensor":
            # the EM loop keeps the GPU busy back to back: the clocks a tensor kernel sees there are the sustained
            # ones (the emission GEMM takes 0.75 ms launched alone and 0.83 ms inside the loop), so the fraction of
            # the measured SUSTAINED peak is printed beside the (judged) fraction of the burst peak
            roof_all[name]["frac_of_sustained_peak"] = ach / (pk["bf16_tflops_sustained"] / 2.0)
        if survey is not None:
            roof_all[name]["survey_bytes"] = survey
    dominant = max((k for k in roof_all), key=lambda k: roof_all[k]["ms"]) if roof_all else None
    roofline = None
    if dominant:
        r = dict(roof_all[dominant])
        r.update({"phase": dominant,
                  "peak_source": pk["src"] + (" HBM copy bandwidth" if r["bound"] == "hbm" else
                                              " bf16 burst / 2 (derived TF32 dense; the phase is timed alone)"),
                  "traffic_source": (NCU_SUMMARY + " (dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set "
                                     "full capture of this kernel at this workload)") if r.get("traffic") else None})
        roofline = r

    # ---- end-to-end through the public API with host buffers (rank-local block; same n_iter per rank)
    e2e = None
    if not args.no_e2e:
        n_iter = args.e2e_iters
        y_host = y_dev.cpu().numpy()
        kw = dict(m_step_maxiter=args.m_step_maxiter, m_step_tol=args.m_step_tol, time_sharded=world > 1)
        # one untimed warm-up call at the same size (pinned staging ring, worker threads, allocator blocks of the
        # result sizes: first-call costs of the process, not of the workload)
        model.fit_em(y_host, key=4, n_iter=2, **kw)
        torch.cuda.synchronize()
        walls = []
        for rep in range(args.e2e_calls):
            barrier()
            t0 = time.perf_counter()
            # the README call: fit_em(y, n_iter=20) with the default random initial posterior (drawn from `key`)
            em = model.fit_em(y_host, key=5 + rep, n_iter=n_iter, **kw)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([wall], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                wall = float(t.item())
            walls.append(wall)
            # bytes actually copied to the host inside the call: every NumPy array of em_res (posterior [T,2,K],
            # its two marginals, params, tuning, histories); entries the reference also keeps on the device
            # (log_posterior_final, saved snapshots: jax arrays there, LazyHostArray here) are not copied
            d2h = sum(int(v.nbytes) for v in em.values() if isinstance(v, np.ndarray))
            d2h += sum(int(a.nbytes) for v in em.values() if isinstance(v, list) for a in v if isinstance(a, np.ndarray))
            del em
        wall = float(np.median(walls))
        e2e = {"value": T_total * n_iter / wall, "unit": UNIT, "h2d_bytes_per_step": int(y_host.nbytes / n_iter),
               "d2h_bytes_per_step": int(d2h / n_iter), "n_iter": n_iter, "wall_s": wall, "wall_s_all": walls,
               "note": "one warm-up call (n_iter=2), then the median of %d timed calls: fit_em(y_host,...) on host "
                       "arrays: H2D of y, n_iter EM iterations, D2H of posterior/posterior_latent_marg/"
                       "posterior_dynamics_marg/params/tuning (the arrays the reference materialises on the host, "
                       "core.py:688-690); bytes are per EM iteration and per rank" % len(walls)}
        del y_host

    # ---- decode throughput (second half of BASELINE.json's metric): device-resident spikes, fitted tuning
    decode = None
    if not args.no_decode and world == 1:
        def timed(fn, reps=3):
            fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps
        tun = m_res[4]
        ms_nb = timed(lambda: model.decode_latent_naive_bayes(y_dev, tuning=tun, return_device=True))
        ms_dec = timed(lambda: model.decode_latent(y_dev, tuning=tun, return_device=True), reps=2)
        decode = {"unit": "bins/s", "naive_bayes": T / (ms_nb * 1e-3), "naive_bayes_ms": ms_nb,
                  "decode_latent": T / (ms_dec * 1e-3), "decode_latent_ms": ms_dec,
                  "note": "decode_latent_naive_bayes / decode_latent (smoother + transition counts) on the bench "
                          "workload, spikes and results resident on the device"}
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        bins = args.cpu_sample_bins or 2000
        rate, parts = cpu_reference_rate(N, K, ls, mv, bins, 1, 0, T)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": 1, "kind": "port",
                        "sample": "1 EM iteration on a %d-bin sample of the workload walked as two reference chunks of "
                                  "%d bins (M-step %.1f s, statistics+E-step %.1f s), extrapolated linearly in T to "
                                  "T=%d; restated reference (NumPy CPU, fp32, reference operation order, BLAS pinned "
                                  "to 1 thread), not JAX"
                                  % (bins, parts["chunk_bins"], parts["t_mstep_s"], parts["t_estep_sample_s"], T)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": "%s: N=%d K=%d, one recording of %d bins time-sharded over %d rank(s) "
                                       "(%d bins per rank, %s scaling), tuning_lengthscale=%g (B=%d), "
                                       "movement_variance=%g, Adam maxiter=%d tol=%g"
                                       % (args.workload, N, K, T_total, world, T_rank, args.scaling, ls, model.n_basis,
                                          mv, args.m_step_maxiter, args.m_step_tol),
                           "parallelism": "time-sharded x%d: neighbour boundary messages (4K floats) per pass, ONE "
                                          "all-reduce per EM iteration (K*(N+1) statistics + log marginal + seam "
                                          "verdict, fp32), replicated M-step" % world,
                           "l2": "inputs larger than L2 (y, ll, alpha, gamma each >= 0.1 GB per rank)",
                           "move_kernel": ("dense custom_transition_kernel exp(-|dx|/150)+0.02, row-normalised; scan = "
                                           "lockstep tcgen05 GEMM per time step over all chains" if dense else
                                           "default RBF, band half width %d" % op.W),
                           "n_chain": loop.es.plan.n_chain, "chunk_len": loop.es.chunk_len,
                           "halo_per_iter": halos, "seam_repairs_on_device_in_timed_region": fixes,
                           "seam_relays_by_host_in_timed_region": relays, "adam_steps_per_iter": n_adam},
                "phases_ms_per_step": per, "phases_host_ms_per_step": phases_host, "roofline": roofline,
                "roofline_all": roof_all, "cpu_baseline": cpu_baseline, "e2e": e2e, "decode": decode,
                "parity_vs_1rank": parity, "tuning_identical_on_all_ranks": tuning_identical,
                "gpu_launches": launches, "clocks": clocks}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="headline", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--bins", type=int, default=0, help="override T (total bins; bins per rank with --scaling weak)")
    ap.add_argument("--m-step-maxiter", type=int, default=1000)
    ap.add_argument("--m-step-tol", type=float, default=1e-6)
    ap.add_argument("--e2e-iters", type=int, default=20)
    ap.add_argument("--e2e-calls", type=int, default=3)
    ap.add_argument("--parity-iters", type=int, default=4)
    ap.add_argument("--cpu-sample-bins", type=int, default=0,
                    help="bins per step of the CPU arm (default: 2000 for the in-line baseline, sized to a ~3 minute "
                         "run for --impl reference)")
    ap.add_argument("--clocks-ms", type=int, default=20, help="nvidia-smi sampling period during the timed region")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-decode", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--phase-steps", type=int, default=None,
                    help="EM iterations of the instrumented (per-phase events) pass after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (float32/float64, at most "
                         "64 MB: T-sized arrays on a fixed, seeded sample of time bins, listed in *bins.npy)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    ClockSampler.PERIOD_MS = max(5, args.clocks_ms)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
