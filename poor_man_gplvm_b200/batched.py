"""Batched callers of the hot path (SURVEY.md section 8(f) row F3).

The reference calls ``decode_latent`` / ``decode_latent_naive_bayes`` hundreds of times on the same spike matrix:
``model_selection_helper.get_downsampled_lml`` (:243-260, n_repeat latent masks), ``get_lml_test_history``
(:424-445, one call per saved tuning) and ``test.shuffle_and_decode`` / ``test_one_model`` (test.py:27-63, n_shuffle
circular shuffles).  Every such call re-uploads the spikes, re-derives the fp16 counts and the lgamma row term, and --
for the ones that only read a log marginal -- runs a backward pass nobody looks at.

Here the recording is prepared once (:class:`DecodeSession`: spikes on the device, emission operands, E-step
buffers) and each variant costs one emission GEMM + one forward scan (``forward_only``) or one full decode.  Same
function names, arguments and result layout as the reference; masks / shuffles are drawn with NumPy generators
(``jax.random.choice(replace=False)`` and the unseeded ``np.random`` of the reference are not reproducible streams),
or passed in explicitly (``latent_masks=``, ``shifts=``) for run-for-run comparisons.
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from .core import _seed_from_key, _unwrap_tsd
from .estep import EStep

# per-bin key of the shuffle test (reference test.py:50-51)
SIG_KEYS = {'naive_bayes': 'log_marginal_l', 'dynamics': 'log_one_step_predictive_marginals_all'}
# device memory of one batch of stacked naive-Bayes shuffles (fp16 counts, lgam and ll of every shuffle in it); at
# most a quarter of the free memory
SHUFFLE_BATCH_BYTES = 16 << 30
# int64 gather index of one neuron slab when the fp32 fallback materialises a rolled matrix
ROLL_INDEX_BYTES = 256 << 20


class DecodeSession:
    """One recording, many decodes: the spikes live on the device, the count-derived emission operands and the scan
    buffers are built once per neuron mask."""

    def __init__(self, model, y, ma_neuron=None, likelihood_scale=1.0, hyperparam={}):
        """ma_neuron: None, [N] or [T,N] (fixed for the session: the count-derived operands depend on it)."""
        self.model = model
        y, self.t_l = _unwrap_tsd(y)
        with _guard(model):
            self.y = model._dev(y)
            self.T = self.y.shape[0]
            _, _, _, _, self.op = model._transition_pack(dict(hyperparam))
            ma_n, _ = model._masks(ma_neuron, None, self.T)
            self.es = EStep(self.y, self.op, ma_n, None, float(likelihood_scale))
        self._yT16 = self._es_shuffle = self._swap = None      # built by the first shuffled() call

    def log_marginal(self, tuning=None, ma_latent=None):
        """log_marginal_final of decode_latent (reference core.py:485) from the forward filter alone."""
        m = self.model
        with _guard(m):
            es = self.es
            es.ma_latent = m._dev(m.ma_latent_default if ma_latent is None else ma_latent)
            res = es.run(m._dev(m.tuning if tuning is None else tuning), forward_only=True)
            return float(res.log_marginal)

    def naive_bayes_total(self, tuning=None, ma_latent=None):
        """log_marginal_total of decode_latent_naive_bayes (reference core.py:520)."""
        m = self.model
        with _guard(m):
            es = self.es
            ma_l = m._dev(m.ma_latent_default if ma_latent is None else ma_latent)
            ll = es.em.loglik(m._dev(m.tuning if tuning is None else tuning), ma_l, 1.0, out=es.ll)
            _, lml = ops.naive_bayes_normalize(ll, inplace=True)
            return float(lml.sum(dtype=torch.float64).item())

    def shuffled(self, shifts, decoder_type, tuning=None, ma_latent=None, max_batch=None, dt_l=1.0):
        """Per-bin key of the shuffle test (reference test.py:27-66) for every row of ``shifts`` [n_shuffle, N]
        (neuron n rolled by shifts[i, n] as np.roll does; a row of zeros is the recording itself): device tensor
        [n_shuffle, T] of ``log_marginal_l`` (naive Bayes, scalar ``dt_l``) or of
        ``log_one_step_predictive_marginals_all`` (dynamics, forward filter only).

        With fp16-exact counts no shuffled matrix is materialised: ``pmg_counts_prepare_shifted`` writes the
        emission operand of the shuffles straight from a neuron-major copy of the session's fp16 counts.  Naive Bayes
        stacks up to ``max_batch`` shuffles along time (default: what fits a fixed memory budget) into one shifted
        prepare, one emission GEMM and one row log-sum-exp; every row equals decode_latent_naive_bayes of the rolled
        matrix bit for bit.  Counts that are not fp16-exact take the fp32 path on each rolled matrix."""
        if decoder_type not in SIG_KEYS:
            raise ValueError("decoder_type %r not supported (naive_bayes or dynamics)" % (decoder_type,))
        _check_shuffle_family(self.model)
        if self.es.em.mode != 0:
            raise ValueError("shuffle tests take ma_neuron None or [N]; the session was built with a [T,N] mask")
        dt = _scalar_dt(dt_l)
        if decoder_type == 'dynamics' and dt != 1.0:
            raise ValueError("dt_l applies to the naive-Bayes decoder only (decode_latent has no bin width)")
        T, N = self.y.shape
        sh = normalize_shifts(shifts, T, N)
        n = sh.shape[0]
        m = self.model
        with _guard(m):
            dev = self.y.device
            tun = m._dev(m.tuning if tuning is None else tuning)
            ma_l = m._dev(m.ma_latent_default if ma_latent is None else ma_latent)
            ma_vec = self.es.em.ma_vec
            out = torch.empty((n, T), dtype=torch.float32, device=dev)
            if n == 0:
                return out
            exact = self.es.em.A16.exact
            if exact:
                if self._yT16 is None:          # neuron-major fp16 counts: each shifted window is contiguous
                    self._yT16 = self.es.em.A16.data[:, :N].t().contiguous()
                sh_dev = torch.from_numpy(sh.astype(np.int32)).to(dev)
            if decoder_type == 'naive_bayes':
                K = tun.shape[0]
                ld16 = (N + 7) // 8 * 8          # the operand of decode_latent_naive_bayes (no column of ones)
                per = T * ((2 * ld16 + 4) if exact else 0) + T * 4 * K
                budget = min(SHUFFLE_BATCH_BYTES, torch.cuda.mem_get_info(dev)[0] // 4)
                b = int(max_batch) if max_batch is not None else max(1, budget // per)
                b = max(1, min(b, n, (ops.EMISSION_MAX_ROWS // T) if exact else 1))
                ll = torch.empty((b * T, K), dtype=torch.float32, device=dev)
                if exact:
                    data = torch.empty((b * T, ld16), dtype=torch.float16, device=dev)
                    lgam = torch.empty(b * T, dtype=torch.float32, device=dev)
                else:
                    rolled = torch.empty_like(self.y)
                ops.phase("setup")
                for i0 in range(0, n, b):
                    nb = min(b, n - i0)
                    if exact:
                        em = _ShiftedOperand(ops.CountsF16Shifted(self._yT16, T, sh_dev[i0:i0 + nb], ld16, ma_vec,
                                                                  data=data, lgam=lgam), ma_vec)
                    else:
                        em = ops.EmissionOperands(_roll_neurons(self.y, sh[i0], rolled), self.es.ma_neuron)
                    ops.phase("shifted_prepare")
                    ll_b = em.loglik(tun, ma_l, dt, out=ll[:nb * T])
                    ops.phase("emission")
                    ops.naive_bayes_lml(ll_b, out=out[i0:i0 + nb].view(-1))
                    ops.phase("logsumexp")
                return out
            # dynamics: one forward filter per shuffle on an E-step whose emission operand is swapped per shuffle
            es = self._shuffle_estep()
            es.ma_latent = ma_l
            if exact:
                ld16 = self.es.em.A16.ld         # the operand of decode_latent
                data = torch.empty((T, ld16), dtype=torch.float16, device=dev)
                lgam = torch.empty(T, dtype=torch.float32, device=dev)
            else:
                rolled = torch.empty_like(self.y)
            ops.phase("setup")
            for i in range(n):
                if exact:
                    self._swap.cur = _ShiftedOperand(ops.CountsF16Shifted(self._yT16, T, sh_dev[i:i + 1], ld16,
                                                                          ma_vec, data=data, lgam=lgam), ma_vec)
                else:
                    self._swap.cur = ops.EmissionOperands(_roll_neurons(self.y, sh[i], rolled), self.es.ma_neuron,
                                                          ones_col=True)
                ops.phase("shifted_prepare")
                res = es.run(tun, forward_only=True)
                out[i].copy_(res.lmr)
                ops.phase("forward")
            self._swap.cur = None
            return out

    def _shuffle_estep(self):
        if self._es_shuffle is None:
            self._swap = _SwapEmission()
            self._es_shuffle = EStep(self.y, self.op, self.es.ma_neuron, None, self.es.scale,
                                     emission_factory=lambda y, ma: self._swap)
        return self._es_shuffle


class _ShiftedOperand:
    """Emission operand of stacked shifted counts: the tensor-core path of EmissionOperands.loglik (mode 0)."""

    def __init__(self, y16, ma_vec):
        self.A16, self.ma_vec = y16, ma_vec

    def loglik(self, tuning, ma_latent=None, dt=1.0, out=None):
        L16, lam_sum = ops.emission_prepare_f16(tuning, self.A16, self.ma_vec, dt)
        return ops.emission_poisson_f16(self.A16, L16, lam_sum, self.A16.lgam, tuning.shape[0], ma_latent, out=out)


class _SwapEmission:
    """Emission hook of the shuffle E-step: delegates to the operand of the shuffle being filtered."""
    mode = 0
    A16 = None               # forward-only passes: no statistics GEMM reads the counts

    def __init__(self):
        self.cur = None

    def loglik(self, tuning, ma_latent=None, dt=1.0, out=None):
        return self.cur.loglik(tuning, ma_latent, dt, out=out)


def _roll_neurons(y, shift_row, out):
    """out[t, n] = y[(t - shift_row[n]) mod T, n] for the fp32 fallback, in neuron slabs whose int64 gather index
    stays within ROLL_INDEX_BYTES."""
    T, N = y.shape
    slab = max(1, min(N, ROLL_INDEX_BYTES // (8 * T)))
    t = torch.arange(T, device=y.device).unsqueeze(1)
    for n0 in range(0, N, slab):
        s = torch.as_tensor(np.asarray(shift_row[n0:n0 + slab], dtype=np.int64), device=y.device)
        out[:, n0:n0 + slab] = torch.gather(y[:, n0:n0 + slab], 0, (t - s.unsqueeze(0)) % T)
    return out


def _guard(model):
    import contextlib
    dev = model.device
    return torch.cuda.device(dev) if dev.type == "cuda" else contextlib.nullcontext()


# ------------------------------------------------------------------------------------------------------------
# model_selection_helper.py
# ------------------------------------------------------------------------------------------------------------
def draw_latent_masks(n_latent_bin, downsample_frac, n_repeat, key=4):
    """n_repeat 0/1 masks with int(K * frac) ones each (reference model_selection_helper.py:249-254; NumPy stream)."""
    rng = np.random.default_rng(_seed_from_key(key))
    n_sel = int(n_latent_bin * downsample_frac)
    masks = np.zeros((n_repeat, n_latent_bin), dtype=np.float32)
    for i in range(n_repeat):
        masks[i, rng.choice(n_latent_bin, size=n_sel, replace=False)] = 1.0
    return masks


def get_downsampled_lml(model_fit, y_test, downsample_frac=0.2, n_repeat=10, key=4, latent_masks=None, **kwargs):
    """reference model_selection_helper.py:243-260: mean / std over n_repeat random latent masks of the log marginal
    of ``decode_latent(y_test, ma_latent=mask)``.  kwargs: tuning, hyperparam, ma_neuron, likelihood_scale (as
    ``decode_latent``).  One emission GEMM + one forward scan per mask on a shared :class:`DecodeSession`."""
    if latent_masks is None:
        latent_masks = draw_latent_masks(model_fit.n_latent_bin, downsample_frac, n_repeat, key)
    ses = DecodeSession(model_fit, y_test, ma_neuron=kwargs.get("ma_neuron"),
                        likelihood_scale=kwargs.get("likelihood_scale", 1.0), hyperparam=kwargs.get("hyperparam", {}))
    lml_l = [ses.log_marginal(tuning=kwargs.get("tuning"), ma_latent=mask) for mask in np.asarray(latent_masks)]
    return {'value': np.mean(lml_l), 'std': np.std(lml_l), 'lml_l': lml_l}


def get_lml_test_history(y_test, model, tuning_saved, do_nb=True, ma_temporal=None):
    """reference model_selection_helper.py:424-445: test log marginal under every saved tuning (naive Bayes total or
    the smoother's log marginal); ``ma_temporal`` [T] expands to a [T,N] neuron mask."""
    ma_neuron = None
    if ma_temporal is not None:
        y_arr, _ = _unwrap_tsd(y_test)
        ma_neuron = np.ones((1, np.shape(y_arr)[1]), np.float32) * np.asarray(ma_temporal, np.float32)[:, None]
    ses = DecodeSession(model, y_test, ma_neuron=ma_neuron)
    fn = ses.naive_bayes_total if do_nb else ses.log_marginal
    return np.array([fn(tuning=tun) for tun in tuning_saved])


# ------------------------------------------------------------------------------------------------------------
# test.py (shuffle tests; not pytest tests)
# ------------------------------------------------------------------------------------------------------------
def draw_shifts(n_time, n_neuron, n_shuffle, seed=None):
    """[n_shuffle, n_neuron] circular shifts in [0, n_time) (the reference draws them with the global np.random)."""
    rng = np.random.default_rng(seed)
    return rng.integers(0, n_time, size=(n_shuffle, n_neuron))


def _roll_columns(y_dev, shift_dev):
    """y_shuffled[t, n] = y[(t - shift[n]) mod T, n]  (np.roll per neuron, reference test.py:22-23)."""
    T = y_dev.shape[0]
    idx = (torch.arange(T, device=y_dev.device).unsqueeze(1) - shift_dev.unsqueeze(0)) % T
    return torch.gather(y_dev, 0, idx)


def circular_shuffle_data(spk_tsdf, n_shuffle=100, ep=None, shifts=None, seed=None, device=None):
    """reference test.py:10-24: every neuron circularly shifted by its own random offset; yields n_shuffle arrays
    (device tensors when the input is one or ``device`` is given, else NumPy)."""
    if ep is not None:
        spk_tsdf = spk_tsdf.restrict(ep)                 # pynapple TsdFrame
    y, _ = _unwrap_tsd(spk_tsdf)
    on_dev = isinstance(y, torch.Tensor) or device is not None
    if on_dev and not isinstance(y, torch.Tensor):
        y = torch.as_tensor(np.asarray(y, dtype=np.float32)).to(device)
    n_time, n_neuron = y.shape
    if shifts is None:
        shifts = draw_shifts(n_time, n_neuron, n_shuffle, seed)
    for i in range(n_shuffle):
        if on_dev:
            yield _roll_columns(y, torch.as_tensor(np.asarray(shifts[i]), device=y.device))
        else:
            out = np.empty_like(np.asarray(y))
            for j in range(n_neuron):
                out[:, j] = np.roll(np.asarray(y)[:, j], int(shifts[i][j]))
            yield out


def shuffle_and_decode(model, spk_tsdf, n_time_per_chunk=10000, dt_l=1, n_shuffle=100, ep=None,
                       decoder_type='naive_bayes', shifts=None, seed=None, keys=None):
    """reference test.py:27-45: decode n_shuffle circular shuffles; every result key stacked over the shuffles.
    The spikes are uploaded once and shuffled on the device.  keys: optional subset of result keys to keep (the
    reference stacks all of them: n_shuffle x T x K floats for the posteriors)."""
    if decoder_type not in ('naive_bayes', 'dynamics'):
        raise ValueError(f"decoder_type {decoder_type} not supported")
    if ep is not None:
        spk_tsdf = spk_tsdf.restrict(ep)
    y, _ = _unwrap_tsd(spk_tsdf)
    with _guard(model):
        y_dev = model._dev(y)
        out = None
        for y_sh in circular_shuffle_data(y_dev, n_shuffle=n_shuffle, shifts=shifts, seed=seed):
            if decoder_type == 'naive_bayes':
                res = model.decode_latent_naive_bayes(y_sh, n_time_per_chunk=n_time_per_chunk, dt_l=dt_l)
            else:
                res = model.decode_latent(y_sh, n_time_per_chunk=n_time_per_chunk)
            if out is None:
                out = {k: [] for k in res if keys is None or k in keys}
            for k in out:
                out[k].append(np.asarray(res[k]))
    return {k: np.array(v) for k, v in out.items()}


def test_one_model(y_true, model_fit, n_shuffle=100, decoder_type='naive_bayes', sig_key=None, seed=None):
    """reference test.py:48-66: per-bin significance of the decode against the 97.5 % quantile over shuffles."""
    y_val, y_t = _unwrap_tsd(y_true)
    if sig_key is None:
        sig_key = 'log_marginal_l' if decoder_type == 'naive_bayes' else 'log_one_step_predictive_marginals_all'
    if decoder_type == 'naive_bayes':
        res_true = model_fit.decode_latent_naive_bayes(y_val)
    elif decoder_type == 'dynamics':
        res_true = model_fit.decode_latent(y_val)
    else:
        raise ValueError(f"decoder_type {decoder_type} not supported")
    res_shuffle = shuffle_and_decode(model_fit, y_val, n_time_per_chunk=10000, dt_l=1, n_shuffle=n_shuffle, ep=None,
                                     decoder_type=decoder_type, seed=seed)
    log_marg_thresh = np.quantile(res_shuffle[sig_key], 0.975, axis=0)
    is_sig = np.asarray(res_true[sig_key]) > log_marg_thresh
    is_sig_tsd = is_sig
    if y_t is not None:
        try:
            import pynapple as nap
            is_sig_tsd = nap.Tsd(d=is_sig, t=y_t)
        except Exception:
            pass
    return {'decode_res_true': res_true, 'decode_res_shuffle': res_shuffle, 'log_marg_thresh': log_marg_thresh,
            'is_sig_tsd': is_sig_tsd}


test_one_model.__test__ = False          # a shuffle test of a model, not a pytest test


def normalize_shifts(shifts, n_time, n_neuron):
    """[n_shuffle, n_neuron] integer shifts -> int64 in [0, n_time): np.mod gives negative shifts and shifts of
    n_time or more the meaning np.roll gives them."""
    s = np.asarray(shifts)
    if s.ndim != 2 or s.shape[1] != n_neuron:
        raise ValueError("shifts must be [n_shuffle, %d], got shape %s" % (n_neuron, s.shape))
    if s.size and not np.issubdtype(s.dtype, np.integer):
        raise ValueError("shifts must be integers, got %s" % s.dtype)
    return np.mod(s.astype(np.int64), int(n_time))


def quantile_rows(x, q):
    """np.quantile(x, q, axis=0) (method 'linear') of a [n, T] float32 tensor, on the tensor's device.  Same
    arithmetic as NumPy on float32 data -- virtual index (n-1)*q, its fraction and the two-sided lerp, all in float32
    -- sorted in column blocks of bounded size."""
    if x.dim() != 2 or x.shape[0] == 0:
        raise ValueError("quantile_rows takes a non-empty [n, T] tensor")
    x = x.to(torch.float32)
    n, T = x.shape
    pos = np.float32(n - 1) * np.float32(q)
    lo = int(np.floor(pos))
    g = np.float32(pos - np.float32(lo))
    hi = min(lo + 1, n - 1)
    out = torch.empty(T, dtype=torch.float32, device=x.device)
    cols = max(1, (1 << 24) // n)
    for c0 in range(0, T, cols):
        s = torch.sort(x[:, c0:c0 + cols], dim=0).values
        a, b = s[lo], s[hi]
        d = b - a
        out[c0:c0 + cols] = (a + d * float(g)) if g < 0.5 else (b - d * float(np.float32(1) - g))
    return out


def _scalar_dt(dt_l):
    dt = np.asarray(dt_l, dtype=np.float64)
    if dt.size != 1:
        raise ValueError("shuffle tests take a scalar dt_l (per-bin dt_l is not supported)")
    dt = float(dt.reshape(()))
    if not dt > 0:
        raise ValueError("dt_l must be positive")
    return dt


def _check_shuffle_family(model):
    from .families import _GPLVM1DBase
    if isinstance(model, _GPLVM1DBase) or model._emission_factory({}) is not None:
        raise ValueError("shuffle_test supports PoissonGPLVMJump1D; %s has a different emission or start message"
                         % type(model).__name__)


def shuffle_test(model_fit, y, n_shuffle=100, decoder_type='naive_bayes', q=0.975, shifts=None, seed=None,
                 tuning=None, ma_neuron=None, ma_latent=None, likelihood_scale=1., dt_l=1., return_device=False,
                 max_batch=None):
    """Significance of every decoded bin against ``n_shuffle`` circular shuffles (reference test.py:27-66 with the
    per-bin key only): the q-quantile over the shuffles of ``log_marginal_l`` (naive Bayes) or
    ``log_one_step_predictive_marginals_all`` (dynamics) is the threshold the unshuffled key must exceed.

    Everything stays on the device until the end: the shuffles are decoded from a neuron-major fp16 copy of the
    counts (see :meth:`DecodeSession.shuffled`), the quantile is taken on the device.  Returns ``sig_key``,
    ``sig_true`` [T], ``sig_shuffle`` [n_shuffle, T] (the reference's ``decode_res_shuffle[sig_key]``),
    ``log_marg_thresh`` [T] and ``is_sig_tsd`` [T] bool (a Tsd when ``y`` is a TsdFrame); NumPy arrays, or device
    tensors with ``return_device=True``.  ``shifts`` [n_shuffle, N] (any integers, np.roll semantics) default to
    :func:`draw_shifts` with ``seed``.  ``dt_l``: scalar bin width of the naive-Bayes decoder."""
    if decoder_type not in SIG_KEYS:
        raise ValueError("decoder_type %r not supported (naive_bayes or dynamics)" % (decoder_type,))
    if not 0.0 < float(q) < 1.0:
        raise ValueError("q must lie in (0, 1), got %r" % (q,))
    _check_shuffle_family(model_fit)
    dt = _scalar_dt(dt_l)
    if ma_neuron is not None and np.ndim(ma_neuron) != 1:
        raise ValueError("shuffle tests take ma_neuron None or [N] (a [T,N] mask does not shift with the counts)")
    y_val, y_t = _unwrap_tsd(y)
    if not isinstance(y_val, torch.Tensor):
        y_val = np.asarray(y_val)
    T, N = tuple(y_val.shape)
    if shifts is None:
        shifts = draw_shifts(T, N, n_shuffle, seed)
    if np.shape(shifts) != (n_shuffle, N):
        raise ValueError("shifts must be [n_shuffle, N] = [%d, %d], got shape %s" % (n_shuffle, N, np.shape(shifts)))
    sh = normalize_shifts(shifts, T, N)
    ses = DecodeSession(model_fit, y_val, ma_neuron=ma_neuron, likelihood_scale=likelihood_scale)
    # row 0: the recording itself, through the same path as the shuffles
    rows = ses.shuffled(np.concatenate([np.zeros((1, N), np.int64), sh]), decoder_type, tuning=tuning,
                        ma_latent=ma_latent, max_batch=max_batch, dt_l=dt)
    sig_true, sig_shuffle = rows[0], rows[1:]
    with _guard(model_fit):
        thresh = quantile_rows(sig_shuffle, q)
        ops.phase("quantile")
        is_sig = sig_true > thresh
    if not return_device:
        sig_true, sig_shuffle, thresh, is_sig = (t.cpu().numpy() for t in (sig_true, sig_shuffle, thresh, is_sig))
        if y_t is not None:
            try:
                import pynapple as nap
                is_sig = nap.Tsd(d=is_sig, t=y_t)
            except Exception:
                pass
    return {'sig_key': SIG_KEYS[decoder_type], 'sig_true': sig_true, 'sig_shuffle': sig_shuffle,
            'log_marg_thresh': thresh, 'is_sig_tsd': is_sig}


shuffle_test.__test__ = False


def compute_entropy(logp_l, axis=(-1, -2)):
    """reference test.py:68-79: -sum p log p over `axis`."""
    logp_l = np.asarray(logp_l)
    with np.errstate(invalid="ignore"):
        term = np.where(np.isneginf(logp_l), 0.0, np.exp(logp_l) * logp_l)      # 0 log 0 = 0 (our logs may be -inf)
    return -np.sum(term, axis=axis)
