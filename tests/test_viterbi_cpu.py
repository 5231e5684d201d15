"""Viterbi oracle against brute-force enumeration, its start convention, the tie rule, and the inputs
decode_latent_viterbi rejects before any device work (no GPU needed)."""
import itertools

import numpy as np
import pytest

from oracle import linear_ref
from oracle import viterbi_ref as vr
from poor_man_gplvm_b200 import gp_kernel as gpk


def _problem(K, T, seed, scale=1.0, masked=None, mv=1.0):
    rng = np.random.default_rng(seed)
    P, logP, M, logM = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), mv, 0.05, 0.2)
    logP = logP.astype(np.float64)
    logP[1] = -np.log(K)          # the jump kernel exactly (the filter of linear_ref uses 1/K)
    ll = rng.normal(0.0, 2.0, size=(T, K))
    if masked is not None:
        ll[:, masked] = -1e20
    return ll, logP, logM, scale


def _all_scores(ll, logP, logM, scale, log_prior0=None):
    T, K = ll.shape
    paths = np.array(list(itertools.product(range(2 * K), repeat=T)), dtype=np.int64)
    scores = np.array([vr.score(p, ll, logP, logM, scale, log_prior0=log_prior0) for p in paths])
    return paths, scores


@pytest.mark.parametrize("K", [2, 3])
@pytest.mark.parametrize("T", [1, 2, 4])
@pytest.mark.parametrize("case", ["plain", "masked_scaled"])
def test_oracle_matches_brute_force(K, T, case):
    masked, scale = (1, 0.7) if case == "masked_scaled" else (None, 1.0)
    ll, logP, logM, s = _problem(K, T, seed=10 * K + T, scale=scale, masked=masked)
    path, lj = vr.viterbi(ll, logP, logM, s)
    paths, scores = _all_scores(ll, logP, logM, s)
    best = int(np.argmax(scores))
    assert abs(lj - scores[best]) <= 1e-12 * abs(scores[best])
    assert abs(vr.score(path, ll, logP, logM, s) - lj) <= 1e-12 * abs(lj)
    np.testing.assert_array_equal(path, paths[best])
    if masked is not None:
        assert not np.any(path % K == masked)
    # the start is marginalised: the sum over all paths is the filter's marginal likelihood
    _, lmr, _ = linear_ref.forward(ll, np.exp(logP[0]), np.exp(logM.astype(np.float64)), s)
    m = scores.max()
    lse = m + np.log(np.exp(scores - m).sum())
    assert abs(lse - lmr.sum()) <= 1e-12 * abs(lmr.sum())


def test_banded_oracle_equals_dense_when_band_covers_every_move():
    ll, logP, logM, s = _problem(6, 9, seed=3)
    p0, l0 = vr.viterbi(ll, logP, logM, s)
    p1, l1 = vr.viterbi(ll, logP, logM, s, band=5)
    np.testing.assert_array_equal(p0, p1)
    assert l0 == l1


@pytest.mark.parametrize("K", [2, 3])
@pytest.mark.parametrize("T", [1, 2, 4])
@pytest.mark.parametrize("band", [None, 1])
def test_exact_ties_pick_the_smallest_flat_index(K, T, band):
    """Small integer log-probabilities make every sum exact, so many paths tie.  Among the optimal paths the
    decoder returns the one that is smallest read from the last bin backwards (smallest final state, then
    smallest predecessor at every step)."""
    rng = np.random.default_rng(100 * K + T)
    for _ in range(20):
        ll = rng.integers(-2, 1, size=(T, K)).astype(np.float64)
        logP = rng.integers(-2, 1, size=(2, K, K)).astype(np.float64)
        logP[1] = -1.0                                      # the jump kernel is constant
        if band is not None:
            far = np.abs(np.arange(K)[:, None] - np.arange(K)[None, :]) > band
            logP[0][far] = -np.inf
        logM = rng.integers(-2, 1, size=(2, 2)).astype(np.float64)
        lp0 = rng.integers(-2, 1, size=(2, K)).astype(np.float64)
        path, lj = vr.viterbi(ll, logP, logM, log_prior0=lp0, band=band)
        paths, scores = _all_scores(ll, logP, logM, 1.0, log_prior0=lp0)
        opt = paths[scores == scores.max()]
        want = min(opt, key=lambda p: tuple(p[::-1]))
        assert lj == scores.max()
        np.testing.assert_array_equal(path, want)


def test_flat_symmetric_problem_decodes_to_state_zero():
    K, T = 5, 4
    _, logP, _, logM = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), 1.0, 0.5, 0.5,
                                                     custom_kernel=np.ones((K, K), np.float32))
    path, _ = vr.viterbi(np.zeros((T, K)), logP, logM)
    np.testing.assert_array_equal(path, np.zeros(T, np.int64))


# ---- inputs rejected before any device work
def _model():
    import poor_man_gplvm_b200 as pmg
    return pmg.PoissonGPLVMJump1D(6, 12, tuning_lengthscale=3.0)


@pytest.mark.parametrize("kw, match", [
    (dict(ma_latent=np.zeros(12, np.float32)), "masks every latent bin"),
    (dict(ma_latent=np.ones(11, np.float32)), "ma_latent must be"),
    (dict(ma_neuron=np.ones(5, np.float32)), "ma_neuron must be"),
    (dict(ma_neuron=np.ones((9, 6), np.float32)), "ma_neuron must be"),
])
def test_decode_latent_viterbi_rejects_bad_masks(kw, match):
    with pytest.raises(ValueError, match=match):
        _model().decode_latent_viterbi(np.zeros((8, 6), np.float32), **kw)


@pytest.mark.parametrize("shape", [(8, 5), (0, 6), (8,)])
def test_decode_latent_viterbi_rejects_bad_counts(shape):
    with pytest.raises(ValueError, match="y must be"):
        _model().decode_latent_viterbi(np.zeros(shape, np.float32))


def test_latent_only_family_rejects_an_empty_latent_mask():
    import poor_man_gplvm_b200 as pmg
    m = pmg.PoissonGPLVM1D(6, 12, tuning_lengthscale=3.0)
    with pytest.raises(ValueError, match="masks every latent bin"):
        m.decode_latent_viterbi(np.zeros((8, 6), np.float32), ma_latent=np.zeros(12, np.float32))
