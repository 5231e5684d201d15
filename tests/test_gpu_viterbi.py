"""Viterbi decoding on the device against the fp64 log-space oracle (oracle/viterbi_ref.py)."""
import numpy as np
import pytest
import torch

import poor_man_gplvm_b200 as pmg
from oracle import viterbi_ref as vr
from poor_man_gplvm_b200 import viterbi
from poor_man_gplvm_b200.estep import EStep
from poor_man_gplvm_b200.families import _GPLVM1DBase
from poor_man_gplvm_b200.synthetic import make_dataset

pytestmark = pytest.mark.gpu
RTOL = 1e-6


def _model(N, K, cls=pmg.PoissonGPLVMJump1D, **kw):
    return cls(N, n_latent_bin=K, tuning_lengthscale=max(2.0, K / 10), **kw)


def _data(T, N, K, seed=0, p_jump=0.01):
    d = make_dataset(T, N, K, seed=seed, p_jump=p_jump)
    return d["y"], d["tuning_true"], d["latent"]


def _run(model, y, tuning, ma_neuron=None, ma_latent=None, scale=1.0, halo=None, chunk_len=None,
         device_repair=True):
    """GPU Viterbi through an EStep (as decode_latent_viterbi builds it) + what the oracle needs."""
    y_dev = model._dev(y)
    P, logP, M, logM, op = model._transition_pack({})
    ma_n, ma_l = model._masks(ma_neuron, ma_latent, y_dev.shape[0])
    carry = op.stationary if isinstance(model, _GPLVM1DBase) else None
    es = EStep(y_dev, op, ma_n, ma_l, scale, halo=halo, chunk_len=chunk_len,
               emission_factory=model._emission_factory({}), carry_in=carry)
    es.device_repair = device_repair
    res = viterbi.run(es, model._dev(tuning))
    path = res.path.cpu().numpy().astype(np.int64)
    return res, path, float(res.log_joint_map.item()), es.ll.cpu().numpy(), logP, logM, \
        (None if carry is None else carry.cpu().numpy()), op


def _check_against_oracle(model, y, tuning, scale=1.0, band=None, **kw):
    res, path, lj, ll, logP, logM, carry, op = _run(model, y, tuning, scale=scale, **kw)
    opath, olj = vr.viterbi(ll, logP, logM, scale, carry=carry, band=band)
    assert abs(lj - olj) <= RTOL * abs(olj), (lj, olj)
    sc = vr.score(path, ll, logP, logM, scale, carry=carry)
    assert abs(sc - olj) <= RTOL * abs(olj), (sc, olj)
    return res, path, opath, op


@pytest.mark.parametrize("K", [7, 64, 400])
@pytest.mark.parametrize("T", [1, 2, 37, 4099])
def test_matches_oracle(K, T):
    y, tun, _ = _data(T, 24, K, seed=K + T)
    _check_against_oracle(_model(24, K), y, tun)


@pytest.mark.parametrize("K", [7, 64, 400])
def test_matches_oracle_long(K):
    T = 200_000
    y, tun, _ = _data(T, 24, K, seed=5)
    m = _model(24, K)
    W = m._transition_pack({})[4].W
    # every move the kernel drops has log P0 < log(1e-11): a jump is always the better way there
    _check_against_oracle(m, y, tun, band=None if K <= 7 else W)


@pytest.mark.parametrize("K", [64, 400])
def test_wide_band_and_scale(K):
    y, tun, _ = _data(4099, 24, K, seed=3)
    m = _model(24, K, movement_variance=20.0)
    assert m._transition_pack({})[4].W > 20
    _check_against_oracle(m, y, tun, scale=0.6)


def test_dense_custom_kernel():
    K = 256
    x = np.arange(K, dtype=np.float32)
    ck = np.exp(-(x[:, None] - x[None, :]) ** 2 / (2 * 40.0 ** 2)).astype(np.float32) + np.float32(1e-3)
    y, tun, _ = _data(4099, 24, K, seed=4)
    m = _model(24, K, custom_transition_kernel=ck)
    op = m._transition_pack({})[4]
    assert op.kind == 1 and op.W == K - 1
    _check_against_oracle(m, y, tun)


def test_masks():
    K, T, N = 64, 4099, 24
    y, tun, _ = _data(T, N, K, seed=6)
    rng = np.random.default_rng(0)
    ma_l = np.ones(K, np.float32)
    ma_l[10:20] = 0
    ma_n = (rng.random((T, N)) > 0.2).astype(np.float32)
    m = _model(N, K)
    res, path, _, _ = _check_against_oracle(m, y, tun, ma_neuron=ma_n, ma_latent=ma_l)
    assert not np.any(ma_l[path % K] == 0)
    _check_against_oracle(m, y, tun, ma_latent=ma_l, ma_neuron=ma_n[0])


def _planted(T=20_000, K=64, N=32):
    y, tun, lat = _data(T, N, K, seed=11)
    return _model(N, K), y, tun, lat


def test_planted_path_is_the_oracle_path():
    m, y, tun, lat = _planted(T=4099)
    res, path, opath, op = _check_against_oracle(m, y, tun)
    np.testing.assert_array_equal(path, opath)
    assert np.mean(np.abs(path % 64 - lat) <= 3) > 0.7


def test_chunking_is_a_no_op():
    m, y, tun, _ = _planted()
    single = _run(m, y, tun, halo=0)
    assert single[0].n_chain == 1
    default = _run(m, y, tun)
    short = _run(m, y, tun, halo=4, chunk_len=64)
    host = _run(m, y, tun, halo=4, chunk_len=64, device_repair=False)
    assert default[0].n_chain > 1 and short[0].n_chain > 100
    assert short[0].n_fix > 0 and host[0].n_relay > 0          # repairs were needed and made
    for r in (default, short, host):
        np.testing.assert_array_equal(r[1], single[1])
        assert abs(r[2] - single[2]) <= RTOL * abs(single[2])


def test_invariants_and_public_api():
    m, y, tun, _ = _planted(T=20_000)
    K = 64
    ma_l = np.ones(K, np.float32)
    ma_l[30:34] = 0
    t_l = np.arange(y.shape[0]) * 0.025
    out = m.decode_latent_viterbi(y, tuning=tun, ma_latent=ma_l, t_l=t_l)
    lat, dyn = np.asarray(getattr(out["map_latent"], "d", out["map_latent"])), \
        np.asarray(getattr(out["map_dynamics"], "d", out["map_dynamics"]))
    assert lat.dtype == np.int64 and dyn.dtype == np.int64 and lat.shape == (y.shape[0],)
    assert set(np.unique(dyn)) <= {0, 1}
    assert not np.any(ma_l[lat] == 0)
    W = m._transition_pack({})[4].W
    moves = dyn[1:] == 0
    assert np.all(np.abs(np.diff(lat))[moves] <= W)
    dec = m.decode_latent(y, tuning=tun, ma_latent=ma_l)
    lm = dec["log_marginal_final"]
    assert out["log_joint_map"] <= lm + 1e-5 * abs(lm)
    # the same decode through the low-level driver
    _, path, lj, *_ = _run(m, y, tun, ma_latent=ma_l)
    np.testing.assert_array_equal(lat, path % K)
    assert lj == out["log_joint_map"]
    dev = m.decode_latent_viterbi(torch.from_numpy(y), tuning=tun, ma_latent=ma_l, return_device=True)
    assert dev["map_latent"].is_cuda and torch.equal(dev["map_latent"].cpu(), torch.from_numpy(lat))


def test_gaussian_jump_family():
    K, N, T = 48, 24, 4099
    _, tun, lat = _data(T, N, K, seed=7)
    rng = np.random.default_rng(1)
    y = (tun[lat] + 0.5 * rng.standard_normal((T, N))).astype(np.float32)
    m = _model(N, K, cls=pmg.GaussianGPLVMJump1D, noise_std=0.5)
    _check_against_oracle(m, y, tun)
    out = m.decode_latent_viterbi(y, tuning=tun)
    assert set(out) == {"map_latent", "map_dynamics", "log_joint_map"}


@pytest.mark.parametrize("cls", [pmg.PoissonGPLVM1D, pmg.GaussianGPLVM1D])
def test_latent_only_families(cls):
    K, N, T = 48, 24, 4099
    y, tun, lat = _data(T, N, K, seed=8, p_jump=0.0)        # no jumps: the smooth prior covers every step
    if cls is pmg.GaussianGPLVM1D:
        y = (tun[lat] + 0.5 * np.random.default_rng(2).standard_normal((T, N))).astype(np.float32)
    m = _model(N, K, cls=cls, movement_variance=3.0)
    res, path, _, _ = _check_against_oracle(m, y, tun)
    assert np.all(path < K)                       # the jump state has probability zero
    out = m.decode_latent_viterbi(y, tuning=tun)
    assert set(out) == {"map_latent", "log_joint_map"}
    np.testing.assert_array_equal(out["map_latent"], path)
    lm = m.decode_latent(y, tuning=tun)["log_marginal_final"]
    assert out["log_joint_map"] <= lm + 1e-5 * abs(lm)


def test_latent_only_underflow_raises_like_decode_latent():
    K, N = 64, 8
    m = pmg.GaussianGPLVM1D(N, n_latent_bin=K, noise_std=0.01, tuning_lengthscale=4.0, movement_variance=1.0)
    tun = np.repeat(np.linspace(0, 20, K, dtype=np.float32)[:, None], N, axis=1)
    y = tun[[0, K - 1]]                           # a jump across the whole track: the smooth prior is zero there
    with pytest.raises(RuntimeError):
        m.decode_latent(y, tuning=tun)
    with pytest.raises(RuntimeError, match="underflowed"):
        m.decode_latent_viterbi(y, tuning=tun)
