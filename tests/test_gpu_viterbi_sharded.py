"""Time-sharded Viterbi decoding (decode_latent_viterbi(time_sharded=True)) against the single-GPU decode and the fp64
oracle.  Workers are spawned as in test_gpu_multirank.py: NCCL with one GPU per rank when there are enough GPUs,
otherwise gloo with every rank on cuda:0, so the whole sharded path -- halo rows, the rank-boundary seam and its host
sweeps, the record all-gather and the cross-rank backtrack -- runs on the real kernels either way."""
import os
import socket

import numpy as np
import pytest

torch = pytest.importorskip("torch")
import torch.multiprocessing as mp

import poor_man_gplvm_b200 as pmg
from oracle import viterbi_ref as vr
from poor_man_gplvm_b200.estep import EStep
from poor_man_gplvm_b200.families import _GPLVM1DBase
from poor_man_gplvm_b200.synthetic import make_dataset

pytestmark = pytest.mark.gpu
RTOL = 1e-6
N, K, T = 32, 64, 20_000


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _model(cls, N, K, dev=None, **kw):
    kw.setdefault("tuning_lengthscale", max(2.0, K / 10))
    return getattr(pmg, cls)(N, n_latent_bin=K, device=dev, **kw)


def _worker(rank, world, port, q, nccl, job):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if nccl else 0)
    torch.cuda.set_device(dev)
    if nccl:
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        lo, hi = job["bounds"][rank], job["bounds"][rank + 1]
        m = _model(job["cls"], job["y"].shape[1], job["K"], dev, **job["model_kw"])
        ma_n = job.get("ma_neuron")
        if ma_n is not None and ma_n.ndim == 2:
            ma_n = ma_n[lo:hi]
        try:
            out = m.decode_latent_viterbi(job["y"][lo:hi], tuning=job["tuning"], ma_neuron=ma_n,
                                          ma_latent=job.get("ma_latent"), likelihood_scale=job.get("scale", 1.0),
                                          time_sharded=True)
            q.put((rank, {"lat": np.asarray(out["map_latent"]), "dyn": out.get("map_dynamics"),
                          "lj": out["log_joint_map"], "info": dict(m._last_estep_info)}))
        except RuntimeError as e:
            q.put((rank, {"error": type(e).__name__, "msg": str(e)}))
    except Exception:  # pragma: no cover
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _sharded(world, job):
    """every rank's result dict, in rank order"""
    nccl = torch.cuda.device_count() >= world
    job.setdefault("bounds", [r * job["y"].shape[0] // world for r in range(world + 1)])
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, nccl, job)) for r in range(world)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=600) for _ in procs)      # a hung rank fails the test here instead of hanging it
    for p in procs:
        p.join(timeout=60)
    for r in range(world):
        assert isinstance(out[r], dict), out[r]
    return [out[r] for r in range(world)]


def _single(job):
    """single-GPU decode_latent_viterbi + the oracle's optimum on the same log-likelihood"""
    m = _model(job["cls"], job["y"].shape[1], job["K"], **job["model_kw"])
    kw = dict(ma_neuron=job.get("ma_neuron"), ma_latent=job.get("ma_latent"), likelihood_scale=job.get("scale", 1.0))
    out = m.decode_latent_viterbi(job["y"], tuning=job["tuning"], **kw)
    y_dev = m._dev(job["y"])
    P, logP, M, logM, op = m._transition_pack({})
    ma_n, ma_l = m._masks(kw["ma_neuron"], kw["ma_latent"], y_dev.shape[0])
    carry = op.stationary if isinstance(m, _GPLVM1DBase) else None
    es = EStep(y_dev, op, ma_n, ma_l, kw["likelihood_scale"], emission_factory=m._emission_factory({}),
               carry_in=carry)
    ll = es.emission(m._dev(job["tuning"])).cpu().numpy()
    carry = None if carry is None else carry.cpu().numpy()
    # K=400: moves outside the kernel's band have log P0 < log(1e-11), a jump is always the better way there
    _, olj = vr.viterbi(ll, logP, logM, kw["likelihood_scale"], carry=carry, band=op.W if job["K"] > 64 else None)
    score = lambda path: vr.score(path, ll, logP, logM, kw["likelihood_scale"], carry=carry)
    return out, olj, score


def _job(cls="PoissonGPLVMJump1D", K=K, T=T, seed=11, p_jump=0.01, **kw):
    d = make_dataset(T, N, K, seed=seed, p_jump=p_jump)
    model_kw = kw.pop("model_kw", {})
    return dict(cls=cls, K=K, y=d["y"], tuning=d["tuning_true"], model_kw=model_kw, lat=d["latent"], **kw)


def _check(job, world):
    """concatenated sharded path == single-GPU path; log_joint_map identical on every rank, and equal to the
    single-GPU value and to the oracle's optimum (also as the oracle's score of the path) within RTOL"""
    single, olj, score = _single(job)
    outs = _sharded(world, job)
    lat = np.concatenate([o["lat"] for o in outs])
    np.testing.assert_array_equal(lat, single["map_latent"])
    flat = lat
    if "map_dynamics" in single:
        dyn = np.concatenate([np.asarray(o["dyn"]) for o in outs])
        np.testing.assert_array_equal(dyn, single["map_dynamics"])
        flat = dyn * job["K"] + lat
    ljs = [o["lj"] for o in outs]
    assert all(v == ljs[0] for v in ljs), ljs
    assert abs(ljs[0] - single["log_joint_map"]) <= RTOL * abs(single["log_joint_map"])
    assert abs(ljs[0] - olj) <= RTOL * abs(olj), (ljs[0], olj)
    sc = score(flat)
    assert abs(sc - olj) <= RTOL * abs(olj), (sc, olj)
    return outs


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_planted_matches_single_gpu(world, monkeypatch):
    monkeypatch.setenv("PMG_HALO", "64")           # many chains per rank at T = 20 000
    outs = _check(_job(), world)
    assert all(o["info"]["n_chain"] > 1 for o in outs)


def test_rank_boundary_seams_repaired_by_host_sweeps(monkeypatch):
    monkeypatch.setenv("PMG_HALO", "4")            # a 4-bin warm-up from the stationary prior misses seam_tol
    outs = _check(_job(), 4)
    assert outs[0]["info"]["relay_fwd_boundary"] == 0
    assert sum(o["info"]["relay_fwd_boundary"] for o in outs[1:]) >= 1
    assert outs[0]["info"]["fix_fwd"] > 0          # interior seams were repaired on the device as well


def _masks(T, K):
    ma_l = np.ones(K, np.float32)
    ma_l[10:14] = 0
    ma_n = (np.random.default_rng(0).random((T, N)) > 0.2).astype(np.float32)
    return ma_l, ma_n


@pytest.mark.parametrize("case", ["K400", "K7", "wide_band", "scale", "masks"])
def test_shapes_and_options(case, monkeypatch):
    """unequal blocks throughout (the middle rank holds most of the recording)"""
    monkeypatch.setenv("PMG_HALO", "64")
    kw = {"K400": dict(K=400), "K7": dict(K=7), "wide_band": dict(model_kw=dict(movement_variance=20.0)),
          "scale": dict(scale=0.6), "masks": {}}[case]
    job = _job(T=12_000, seed=13, **kw)
    if case == "masks":
        job["ma_latent"], job["ma_neuron"] = _masks(12_000, K)
    if case == "wide_band":
        assert _model("PoissonGPLVMJump1D", N, K, **job["model_kw"])._transition_pack({})[4].W > 20
    job["bounds"] = [0, 1500, 9000, 12_000]
    outs = _check(job, 3)
    if case == "masks":
        lat = np.concatenate([o["lat"] for o in outs])
        assert not np.any(job["ma_latent"][lat] == 0)


def test_gaussian_jump_family(monkeypatch):
    monkeypatch.setenv("PMG_HALO", "64")
    job = _job(cls="GaussianGPLVMJump1D", K=48, T=8000, seed=7, model_kw=dict(noise_std=0.5))
    job["y"] = (job["tuning"][job["lat"]] + 0.5 * np.random.default_rng(1).standard_normal(job["y"].shape)
                ).astype(np.float32)
    _check(job, 2)


def test_latent_only_family(monkeypatch):
    monkeypatch.setenv("PMG_HALO", "64")
    job = _job(cls="PoissonGPLVM1D", K=48, T=8000, seed=8, p_jump=0.0, model_kw=dict(movement_variance=3.0))
    outs = _check(job, 3)
    assert all(o["dyn"] is None for o in outs)


@pytest.mark.parametrize("jump_at", [150, 450])
def test_latent_only_underflow_raises_on_every_rank(jump_at):
    """a jump across the whole track, which the smooth prior cannot follow: inside rank 0's block the right rank's
    boundary seam never passes (SeamError after the sweeps), inside rank 1's the global log_joint_map is not finite;
    either way every rank raises the same RuntimeError and none hangs"""
    Kl, Nl = 64, 8
    tun = np.repeat(np.linspace(0, 20, Kl, dtype=np.float32)[:, None], Nl, axis=1)
    y = tun[np.where(np.arange(600) < jump_at, 0, Kl - 1)]
    job = dict(cls="GaussianGPLVM1D", K=Kl, y=y, tuning=tun,
               model_kw=dict(noise_std=0.01, tuning_lengthscale=4.0, movement_variance=1.0))
    with pytest.raises(RuntimeError, match="underflowed"):
        _model(job["cls"], Nl, Kl, **job["model_kw"]).decode_latent_viterbi(y, tuning=tun)
    outs = _sharded(2, job)
    for o in outs:
        assert o.get("error") == "RuntimeError" and "underflowed" in o["msg"], o


def test_single_device_unchanged():
    """time_sharded=True without a process group (world 1) is the single-device decode, bit for bit"""
    job = _job(T=4099, seed=5)
    m = _model(job["cls"], N, K)
    a = m.decode_latent_viterbi(job["y"], tuning=job["tuning"])
    b = m.decode_latent_viterbi(job["y"], tuning=job["tuning"], time_sharded=True)
    for k in ("map_latent", "map_dynamics"):
        np.testing.assert_array_equal(a[k], b[k])
    assert a["log_joint_map"] == b["log_joint_map"]
    assert m._last_estep_info["relay_fwd_boundary"] == 0
