"""bench.py end to end on the GPU at a small size: --steps sets the number of timed EM iterations, and
--dump-outputs writes the results of the last one, identically for two runs with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, cwd):
    # session shape (N=200, K=100) at T=2e5: more bins than the dump budget holds, so the bin sample is exercised
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "session", "--bins", "200000",
           "--steps", "3", "--warmup", "1", "--phase-steps", "0", "--no-e2e", "--no-decode", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=str(cwd), timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_bench_steps_and_dump_outputs(tmp_path):
    line, a = _bench(tmp_path / "a", tmp_path)
    assert line["steps"] == 3 and len(line["config"]["adam_steps_per_iter"]) == 3
    assert set(a) == {"tuning", "params", "log_marginal", "m_step_n_iter", "m_step_final", "m_step_loss_history",
                      "m_step_error_history", "posterior_latent_marg", "posterior_bins"}
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    K, N = 100, 200
    bins = a["posterior_bins"]
    assert a["tuning"].shape == (K, N) and np.all(a["tuning"] > 0)
    assert 0 < len(bins) < 200000 and np.all(np.diff(bins) > 0) and a["posterior_latent_marg"].shape == (len(bins), K)
    # hi + lo pieces of the posterior: a distribution over the latent bins in every sampled time bin
    assert np.max(np.abs(a["posterior_latent_marg"].sum(axis=1) - 1.0)) < 1e-4
    assert a["m_step_loss_history"].shape == (int(a["m_step_n_iter"]),) and np.isfinite(a["log_marginal"])
    _, b = _bench(tmp_path / "b", tmp_path)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
