"""Shuffle significance test on the device (poor_man_gplvm_b200.test.shuffle_test): the shifted count preparation
and the log-marginal-only naive-Bayes pass against the existing kernels, and every shuffle against the single-call
decode of the np.roll'ed matrix."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from poor_man_gplvm_b200.synthetic import make_dataset

pytestmark = pytest.mark.gpu


def _ulp(v):
    return np.spacing(np.abs(np.asarray(v, np.float32)))


def _roll(y, shift_row):
    return np.stack([np.roll(y[:, j], int(shift_row[j])) for j in range(y.shape[1])], axis=1)


def _shifts(T, N, n, seed):
    rng = np.random.default_rng(seed)
    s = rng.integers(-2 * T, 3 * T, size=(n, N))
    s[0, 0] = 0
    s[-1, -1] = T - 1
    if N > 1:
        s[0, 1] = -1
        s[-1, 0] = T + 3
    return s


# ----------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("N", [1, 7, 24, 500, 1003, 3000])
@pytest.mark.parametrize("T", [1, 2, 37, 4099])
def test_counts_prepare_shifted_matches_counts_prepare_on_rolled(N, T):
    from poor_man_gplvm_b200 import batched, ops
    rng = np.random.default_rng(N * 7919 + T)
    y = rng.poisson(1.5, size=(T, N)).astype(np.float32)
    big = rng.random((T, N)) < 0.02                         # counts past the lgamma table, up to the fp16 limit
    y[big] = rng.integers(7, 2049, size=int(big.sum()))
    y_dev = torch.from_numpy(y).cuda()
    src = ops.CountsF16(y_dev, ma_vec=None, want_lgam=True)
    assert src.exact
    yT16 = src.data[:, :N].t().contiguous()
    ma = np.ones(N, np.float32)
    ma[::3] = 0.0
    for ma_vec in (None, torch.from_numpy(ma).cuda()):
        for n_shift in (1, 3):
            raw = _shifts(T, N, n_shift, seed=N + T + n_shift)
            sh = torch.from_numpy(batched.normalize_shifts(raw, T, N).astype(np.int32)).cuda()
            got = ops.CountsF16Shifted(yT16, T, sh, src.ld, ma_vec)
            assert got.T == n_shift * T and got.data.shape == (n_shift * T, src.ld)
            for b in range(n_shift):
                rolled = torch.stack([torch.roll(y_dev[:, j], int(raw[b, j])) for j in range(N)], dim=1).contiguous()
                want = ops.CountsF16(rolled, ma_vec=ma_vec, want_lgam=True)
                assert torch.equal(got.data[b * T:(b + 1) * T], want.data), (b, ma_vec is None)
                assert torch.equal(got.lgam[b * T:(b + 1) * T], want.lgam), (b, ma_vec is None)


@pytest.mark.parametrize("K", [1, 64, 400])
def test_naive_bayes_lml_matches_normalize(K):
    from poor_man_gplvm_b200 import ops
    rng = np.random.default_rng(K)
    T = 3001
    ll = (rng.standard_normal((T, K)) * 30 - 200).astype(np.float32)
    if K > 1:
        ll[:, rng.random(K) < 0.3] = -1e20                 # ma_latent zeros (reference decoder.py:46)
    ll[5] = -1e20                                           # a bin with every latent masked
    ll_dev = torch.from_numpy(ll).cuda()
    _, want = ops.naive_bayes_normalize(ll_dev)
    assert torch.equal(ops.naive_bayes_lml(ll_dev), want)
    _, want2, _ = ops.naive_bayes_normalize(ll_dev, want_post=True)
    assert torch.equal(want2, want)


# ----------------------------------------------------------------------------- end to end
@pytest.fixture(scope="module")
def fitted():
    import poor_man_gplvm_b200 as pmg
    N, K, T = 24, 64, 400
    d = make_dataset(T, N, K, seed=31)
    m = pmg.PoissonGPLVMJump1D(N, K, tuning_lengthscale=8.0)
    m.fit_em(d["y"], key=2, n_iter=4, m_step_maxiter=25, m_step_tol=-1, save_every=2)
    return d["y"].astype(np.float32), m


@pytest.mark.parametrize("max_batch", [1, 2, None])
def test_naive_bayes_rows_equal_single_decodes(fitted, max_batch):
    from poor_man_gplvm_b200 import test as shuf
    y, m = fitted
    T, N = y.shape
    shifts = _shifts(T, N, 5, seed=11)
    ma_n = np.ones(N, np.float32)
    ma_n[3] = ma_n[10] = 0.0
    for kw in (dict(), dict(dt_l=0.37), dict(ma_neuron=ma_n)):
        res = shuf.shuffle_test(m, y, n_shuffle=5, shifts=shifts, max_batch=max_batch, **kw)
        assert res["sig_key"] == "log_marginal_l" and res["sig_shuffle"].shape == (5, T)
        assert np.array_equal(res["sig_true"], m.decode_latent_naive_bayes(y, **kw)["log_marginal_l"])
        for i in range(5):
            want = m.decode_latent_naive_bayes(_roll(y, shifts[i]), **kw)["log_marginal_l"]
            assert np.array_equal(res["sig_shuffle"][i], want), (i, kw)


def test_naive_bayes_threshold_and_flags(fitted):
    from poor_man_gplvm_b200 import test as shuf
    y, m = fitted
    for q in (0.975, 0.5):
        res = shuf.shuffle_test(m, y, n_shuffle=9, seed=4, q=q)
        np_thresh = np.quantile(res["sig_shuffle"], q, axis=0)
        margin = 2 * _ulp(np.maximum(np.abs(np_thresh), np.abs(res["log_marg_thresh"])))
        assert np.all(np.abs(res["log_marg_thresh"] - np_thresh) <= margin)
        clear = np.abs(res["sig_true"] - np_thresh) > margin
        assert res["is_sig_tsd"].dtype == bool and res["is_sig_tsd"].shape == (y.shape[0],)
        assert np.array_equal(res["is_sig_tsd"][clear], (res["sig_true"] > np_thresh)[clear])
    dev = shuf.shuffle_test(m, y, n_shuffle=9, seed=4, return_device=True)
    assert dev["sig_shuffle"].is_cuda and dev["is_sig_tsd"].dtype == torch.bool


def _check_dynamics_row(got, want_lmr, want_lml):
    want_lmr = np.asarray(want_lmr)
    assert np.all(np.abs(got - want_lmr) <= 1e-4 + 2 * _ulp(want_lmr))
    assert np.isclose(got.astype(np.float64).sum(), want_lml, rtol=2e-6)


def test_dynamics_rows_match_single_decodes(fitted):
    from poor_man_gplvm_b200 import test as shuf
    y, m = fitted
    T, N = y.shape
    shifts = _shifts(T, N, 3, seed=12)
    res = shuf.shuffle_test(m, y, n_shuffle=3, shifts=shifts, decoder_type='dynamics')
    assert res["sig_key"] == "log_one_step_predictive_marginals_all" and res["sig_shuffle"].shape == (3, T)
    one = m.decode_latent(y)
    _check_dynamics_row(res["sig_true"], one["log_one_step_predictive_marginals_all"], one["log_marginal_final"])
    for i in range(3):
        one = m.decode_latent(_roll(y, shifts[i]))
        _check_dynamics_row(res["sig_shuffle"][i], one["log_one_step_predictive_marginals_all"],
                            one["log_marginal_final"])


def test_fallback_for_counts_not_exact_in_fp16(fitted):
    from poor_man_gplvm_b200 import test as shuf
    y, m = fitted
    T, N = y.shape
    yf = y + np.float32(0.1)                                 # not representable in fp16: fp32 emission path
    shifts = _shifts(T, N, 3, seed=13)
    res = shuf.shuffle_test(m, yf, n_shuffle=3, shifts=shifts, dt_l=0.8)
    for i in range(3):
        want = m.decode_latent_naive_bayes(_roll(yf, shifts[i]), dt_l=0.8)["log_marginal_l"]
        assert np.array_equal(res["sig_shuffle"][i], want)
    dyn = shuf.shuffle_test(m, yf, n_shuffle=2, shifts=shifts[:2], decoder_type='dynamics')
    for i in range(2):
        one = m.decode_latent(_roll(yf, shifts[i]))
        _check_dynamics_row(dyn["sig_shuffle"][i], one["log_one_step_predictive_marginals_all"],
                            one["log_marginal_final"])


def test_session_rejects_a_time_varying_neuron_mask(fitted):
    from poor_man_gplvm_b200.batched import DecodeSession
    y, m = fitted
    ses = DecodeSession(m, y, ma_neuron=np.ones(y.shape, np.float32))
    with pytest.raises(ValueError, match="mask"):
        ses.shuffled(np.zeros((1, y.shape[1]), np.int64), 'naive_bayes')
