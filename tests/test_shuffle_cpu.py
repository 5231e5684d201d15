"""Host side of the shuffle significance test (poor_man_gplvm_b200.test.shuffle_test): shift normalisation, the
quantile helper against np.quantile, and the inputs it rejects before any device work."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from poor_man_gplvm_b200 import batched


def _ulps(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))


def test_normalize_shifts_has_np_roll_semantics():
    rng = np.random.default_rng(0)
    T, N = 37, 6
    raw = rng.integers(-3 * T, 3 * T, size=(4, N))
    raw[0] = [0, T - 1, -1, T, 2 * T + 5, -T]
    sh = batched.normalize_shifts(raw, T, N)
    assert sh.dtype == np.int64 and sh.min() >= 0 and sh.max() < T
    y = rng.integers(0, 9, size=(T, N))
    for i in range(raw.shape[0]):
        for n in range(N):
            assert np.array_equal(np.roll(y[:, n], int(raw[i, n])), np.roll(y[:, n], int(sh[i, n])))
    with pytest.raises(ValueError):
        batched.normalize_shifts(raw[:, :-1], T, N)
    with pytest.raises(ValueError):
        batched.normalize_shifts(raw[0], T, N)
    with pytest.raises(ValueError):
        batched.normalize_shifts(raw.astype(np.float64) + 0.5, T, N)


@pytest.mark.parametrize("n_shuffle", [1, 2, 3, 8, 100, 101])
@pytest.mark.parametrize("q", [0.975, 0.5, 0.025, 0.9, 0.3, 0.999])
def test_quantile_rows_matches_np_quantile(n_shuffle, q):
    rng = np.random.default_rng(n_shuffle)
    x = (rng.standard_normal((n_shuffle, 5003)) * 40 - 300).astype(np.float32)
    x[:, :7] = -1e20                                   # masked bins of a log marginal: ties at a huge magnitude
    got = batched.quantile_rows(torch.from_numpy(x), q).numpy()
    want = np.quantile(x, q, axis=0)
    assert got.dtype == np.float32 and got.shape == (5003,)
    assert _ulps(got, want).max() <= 2


def test_quantile_rows_column_blocks():
    # more columns than one sort block holds: the blocks must tile the columns exactly
    rng = np.random.default_rng(5)
    x = rng.standard_normal((4096, 4100)).astype(np.float32)
    got = batched.quantile_rows(torch.from_numpy(x), 0.975).numpy()
    assert _ulps(got, np.quantile(x, 0.975, axis=0)).max() <= 2


def test_shuffle_test_rejects_unsupported_inputs():
    import poor_man_gplvm_b200 as pmg
    from poor_man_gplvm_b200 import test as shuf
    N, K, T = 6, 16, 50
    m = pmg.PoissonGPLVMJump1D(N, K)
    y = np.random.default_rng(0).poisson(1.0, size=(T, N)).astype(np.float32)
    with pytest.raises(ValueError, match="decoder_type"):
        shuf.shuffle_test(m, y, n_shuffle=2, decoder_type='other')
    with pytest.raises(ValueError, match="shifts"):
        shuf.shuffle_test(m, y, n_shuffle=2, shifts=np.zeros((3, N), np.int64))
    with pytest.raises(ValueError, match="shifts"):
        shuf.shuffle_test(m, y, n_shuffle=2, shifts=np.zeros((2, N + 1), np.int64))
    for q in (0.0, 1.0, -0.5, 1.5):
        with pytest.raises(ValueError, match="q must"):
            shuf.shuffle_test(m, y, n_shuffle=2, q=q)
    with pytest.raises(ValueError, match="scalar dt_l"):
        shuf.shuffle_test(m, y, n_shuffle=2, dt_l=np.full(T, 0.5))
    with pytest.raises(ValueError, match="positive"):
        shuf.shuffle_test(m, y, n_shuffle=2, dt_l=0.0)
    with pytest.raises(ValueError, match="ma_neuron"):
        shuf.shuffle_test(m, y, n_shuffle=2, ma_neuron=np.ones((T, N), np.float32))
    for fam in (pmg.GaussianGPLVMJump1D(N, K), pmg.PoissonGPLVM1D(N, K), pmg.GaussianGPLVM1D(N, K)):
        with pytest.raises(ValueError, match="PoissonGPLVMJump1D"):
            shuf.shuffle_test(fam, y, n_shuffle=2)
