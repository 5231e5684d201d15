"""Operator layer: PyTorch tensors in, C-ABI calls on the current CUDA stream.

PyTorch is used only for device memory and streams.  Every function here
launches the hand-written sm_100a kernels of libpmgplvm_b200.so; nothing falls
back to torch ops or to the CPU.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib
from ._lib import PmgScanPlan, PmgTransition, check


LAUNCHES = 0          # kernels of libpmgplvm_b200.so launched so far (bench.py reports the delta)
PHASE_HOOK = None     # optional callable(name): bench.py records CUDA events between phases


def _count(n):
    global LAUNCHES
    LAUNCHES += n


def phase(name):
    if PHASE_HOOK is not None:
        PHASE_HOOK(name)


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream():
    """cudaStream_t of torch's current stream on the current device.  Every operator call needs it, ~16 times per EM
    iteration: the raw getter costs ~1 us, building a torch.cuda.Stream object ~10 us -- at 125 000 bins per rank the
    launching thread, not the GPU, was the bottleneck."""
    if _raw_stream is not None:
        return C.c_void_p(_raw_stream(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def _f32(t, name, ndim=None):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError("%s must be a CUDA tensor" % name)
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32, got %s" % (name, t.dtype))
    if ndim is not None and t.dim() != ndim:
        raise ValueError("%s must have %d dims, got shape %s" % (name, ndim, tuple(t.shape)))
    if not t.is_contiguous():
        raise ValueError("%s must be contiguous" % name)
    return t


# ----------------------------------------------------------------------------- emission
def emission_prepare(tuning, ma_neuron=None, dt=1.0):
    """loglam[K,N] = ma*log(tuning*dt+1e-20), lam_sum[K] (reference decoder.py:39-43)."""
    lib = _lib.load()
    _f32(tuning, "tuning", 2)
    K, N = tuning.shape
    if ma_neuron is not None:
        _f32(ma_neuron, "ma_neuron", 1)
    loglam = torch.empty_like(tuning)
    lam_sum = torch.empty(K, dtype=torch.float32, device=tuning.device)
    check(lib.pmg_emission_prepare(K, N, _p(tuning), _p(ma_neuron), float(dt), _p(loglam), _p(lam_sum), _stream()),
          "pmg_emission_prepare")
    _count(1)
    return loglam, lam_sum


def lgamma_rowsum(y, ma_neuron=None, want_ysum=False):
    """lgam[t] = sum_n m lgamma(y+1) (and optionally ysum[t] = sum_n m y); m: None, [N] or [T,N]."""
    lib = _lib.load()
    _f32(y, "y", 2)
    T, N = y.shape
    out = torch.empty(T, dtype=torch.float32, device=y.device)
    ysum = torch.empty(T, dtype=torch.float32, device=y.device) if want_ysum else None
    ldm = 0
    if ma_neuron is not None:
        _f32(ma_neuron, "ma_neuron")
        if ma_neuron.dim() == 2:
            if tuple(ma_neuron.shape) != (T, N):
                raise ValueError("ma_neuron must be [N] or [T,N]")
            ldm = N
        elif ma_neuron.shape[0] != N:
            raise ValueError("ma_neuron must be [N] or [T,N]")
    check(lib.pmg_emission_row_terms(T, N, _p(y), N, _p(ma_neuron), ldm, _p(out), _p(ysum), _stream()),
          "pmg_emission_row_terms")
    _count(1)
    return (out, ysum) if want_ysum else out


def emission_poisson(y, loglam, lam_sum, lgam, ma_latent=None, out=None):
    """ll[T,K] from fp32 operands on CUDA-core tiles (reference decoder.py:30-48,60-71)."""
    lib = _lib.load()
    _f32(y, "y", 2); _f32(loglam, "loglam", 2)
    T, N = y.shape
    K = loglam.shape[0]
    if loglam.shape[1] != N:
        raise ValueError("y has %d neurons but tuning has %d" % (N, loglam.shape[1]))
    if out is None:
        out = torch.empty((T, K), dtype=torch.float32, device=y.device)
    check(lib.pmg_emission_poisson(T, N, K, _p(y), N, _p(loglam), _p(lam_sum), _p(lgam), _p(ma_latent),
                                   _p(out), K, _stream()), "pmg_emission_poisson")
    _count(1)
    return out


class CountsF16:
    """fp16 copy of the spike counts for the tensor-core kernels ([T, ld16], zero padded)."""

    def __init__(self, y, ones_col=False, ma_vec=None, want_lgam=False, want_ysum=False):
        """ones_col: append a column of ones (index N) so that the statistics GEMM also returns sum_t gamma
        (reference fit_tuning_helper.py:41) as column N of its output; the emission GEMM multiplies it by the
        zero padding of its right-hand operand.
        want_lgam: the same pass over the counts also produces ``self.lgam`` [T] = sum_n m_n lgamma(y+1)
        (and ``self.ysum`` with want_ysum) for the neuron mask vector ``ma_vec`` (None = all ones)."""
        lib = _lib.load()
        _f32(y, "y", 2)
        self.T, self.N = y.shape
        self.ones_col = bool(ones_col)
        self.ld = (self.N + (1 if ones_col else 0) + 7) // 8 * 8   # 16-byte rows (TMA); wider padding did not pay
        self.data = torch.empty((self.T, self.ld), dtype=torch.float16, device=y.device)
        self._inexact = torch.zeros(1, dtype=torch.int32, device=y.device)
        self.lgam = self.ysum = None
        if want_lgam:
            if ma_vec is not None:
                _f32(ma_vec, "ma_neuron", 1)
                if ma_vec.shape[0] != self.N:
                    raise ValueError("ma_neuron must be [N]")
            self.lgam = torch.empty(self.T, dtype=torch.float32, device=y.device)
            self.ysum = torch.empty(self.T, dtype=torch.float32, device=y.device) if want_ysum else None
            check(lib.pmg_counts_prepare(self.T, self.N, _p(y), y.stride(0), _p(ma_vec), _p(self.data), self.ld,
                                         int(self.ones_col), _p(self._inexact), _p(self.lgam), _p(self.ysum),
                                         _stream()), "pmg_counts_prepare")
            _count(1)
        else:
            check(lib.pmg_counts_to_f16(self.T, self.N, _p(y), self.N, _p(self.data), self.ld, _p(self._inexact),
                                        _stream()), "pmg_counts_to_f16")
            _count(1)
            if ones_col:
                self.data[:, self.N] = 1.0
        self._exact = None

    @property
    def exact(self):
        """True when every count is exactly representable in fp16 (integers up to 2048)."""
        if self._exact is None:
            self._exact = int(self._inexact.item()) == 0
        return self._exact


class CountsF16Shifted:
    """The fp16 operand and lgamma row term of ``CountsF16(want_lgam=True)`` for ``n_shift`` circular shuffles of the
    same counts, stacked along time: row ``b*T + t`` holds bin t of shuffle b (np.roll of neuron n by
    ``shifts[b, n]``).  Same attributes as CountsF16 (``T`` = n_shift * T rows), so the emission GEMM takes it as is;
    bit-identical to CountsF16 of each rolled fp32 matrix."""
    ones_col = False
    exact = True          # a circular shift keeps each neuron's values: exact whenever the unshifted counts are

    def __init__(self, yT16, T, shifts, ld16, ma_vec=None, data=None, lgam=None):
        """yT16: [N, >=T] fp16, the fp16-exact counts in neuron-major layout; shifts: int32 [n_shift, N] on the
        device, each in [0, T).  data / lgam: optional buffers of at least n_shift*T rows (views are taken)."""
        lib = _lib.load()
        if not (isinstance(yT16, torch.Tensor) and yT16.is_cuda and yT16.dtype == torch.float16 and yT16.dim() == 2
                and (yT16.stride(1) == 1 or yT16.shape[1] == 1)):
            raise TypeError("yT16 must be a row-major [N, T] float16 CUDA tensor")
        self.N = yT16.shape[0]
        if (not isinstance(shifts, torch.Tensor) or shifts.dtype != torch.int32 or shifts.dim() != 2
                or shifts.shape[1] != self.N or not shifts.is_contiguous()):
            raise ValueError("shifts must be a contiguous int32 [n_shift, %d] tensor" % self.N)
        if yT16.shape[1] < T:
            raise ValueError("yT16 has %d time bins, fewer than T=%d" % (yT16.shape[1], T))
        self.n_shift = shifts.shape[0]
        self.T = self.n_shift * int(T)
        self.ld = int(ld16)
        if ma_vec is not None:
            _f32(ma_vec, "ma_neuron", 1)
            if ma_vec.shape[0] != self.N:
                raise ValueError("ma_neuron must be [N]")
        dev = yT16.device
        self.data = (torch.empty((self.T, self.ld), dtype=torch.float16, device=dev) if data is None
                     else data[:self.T])
        self.lgam = torch.empty(self.T, dtype=torch.float32, device=dev) if lgam is None else lgam[:self.T]
        self.ysum = None
        check(lib.pmg_counts_prepare_shifted(int(T), self.N, self.n_shift, _p(yT16), yT16.stride(0), _p(shifts),
                                             _p(ma_vec), _p(self.data), self.ld, _p(self.lgam), _stream()),
              "pmg_counts_prepare_shifted")
        _count(1)


def emission_tile_n(K):
    return int(_lib.load().pmg_emission_tile_n(int(K)))


def emission_prepare_f16(tuning, y16, ma_neuron=None, dt=1.0):
    """(loglam16 [2,Kpad,ld16] fp16 hi/lo pieces, lam_sum[K]).  The two buffers belong to `y16` and are reused by
    every call with the same K (an EM iteration consumes them before the next one rewrites them, in stream order)."""
    lib = _lib.load()
    _f32(tuning, "tuning", 2)
    K, N = tuning.shape
    if N != y16.N:
        raise ValueError("y has %d neurons but tuning has %d" % (y16.N, N))
    cache = getattr(y16, "_prep", None)
    if cache is not None and cache[0] == K and cache[1].device == tuning.device:
        _, L16, lam_sum, Kpad = cache
    else:
        bn = emission_tile_n(K)
        Kpad = (K + bn - 1) // bn * bn
        L16 = torch.empty((2, Kpad, y16.ld), dtype=torch.float16, device=tuning.device)
        lam_sum = torch.empty(K, dtype=torch.float32, device=tuning.device)
        y16._prep = (K, L16, lam_sum, Kpad)
    check(lib.pmg_emission_prepare_f16(K, N, _p(tuning), _p(ma_neuron), float(dt), Kpad, y16.ld, _p(L16),
                                       _p(lam_sum), _stream()), "pmg_emission_prepare_f16")
    _count(1)
    return L16, lam_sum


EMISSION_MAX_ROWS = (1 << 31) - 256     # time bins of one pmg_emission_poisson_f16 call


def emission_poisson_f16(y16, L16, lam_sum, lgam, K, ma_latent=None, out=None):
    """ll[T,K] on the tensor cores (tcgen05 kind::f16, fp32 accumulation)."""
    lib = _lib.load()
    if out is None:
        out = torch.empty((y16.T, K), dtype=torch.float32, device=L16.device)
    check(lib.pmg_emission_poisson_f16(y16.T, y16.N, K, _p(y16.data), y16.ld, _p(L16), L16.shape[1], _p(lam_sum),
                                       _p(lgam), _p(ma_latent), _p(out), out.stride(0), _stream()),
          "pmg_emission_poisson_f16")
    _count(1)
    return out


def emission(y, tuning, lgam, ma_neuron=None, ma_latent=None, dt=1.0, out=None, y16=None, impl=0):
    """Dispatch: tensor cores when the counts are fp16-exact (impl=0), else / impl=1 the fp32 tiles."""
    if impl == 0 and y16 is not None and y16.exact:
        L16, lam_sum = emission_prepare_f16(tuning, y16, ma_neuron, dt)
        return emission_poisson_f16(y16, L16, lam_sum, lgam, tuning.shape[0], ma_latent, out=out)
    loglam, lam_sum = emission_prepare(tuning, ma_neuron, dt)
    return emission_poisson(y, loglam, lam_sum, lgam, ma_latent, out=out)


def emission_prepare_aug(tuning, mode, ma_neuron=None, dt=1.0, rows_out=None):
    """Augmented right-hand operand (see pmg_emission_prepare_aug): mode 1 = [T,N] neuron mask,
    mode 2 = per-bin dt.  Returns (B_aug [rows_out, N_aug] fp32, lam_sum [K])."""
    lib = _lib.load()
    _f32(tuning, "tuning", 2)
    K, N = tuning.shape
    n_aug = 2 * N if mode == 1 else N + 1
    rows = K if rows_out is None else int(rows_out)
    B = torch.empty((rows, n_aug), dtype=torch.float32, device=tuning.device)
    lam_sum = torch.empty(K, dtype=torch.float32, device=tuning.device)
    check(lib.pmg_emission_prepare_aug(K, N, _p(tuning), _p(ma_neuron), float(dt), int(mode), rows, _p(B), n_aug,
                                       _p(lam_sum), _stream()), "pmg_emission_prepare_aug")
    _count(1)
    return B, lam_sum


class EmissionOperands:
    """Left-hand operand and row terms of the emission GEMM for one recording (constant across EM
    iterations), covering the reference's whole mask surface:
      * ma_neuron None / [N]   : A = y, the mask is folded into the right-hand operand (decoder.py:43);
      * ma_neuron [T,N]        : A = [m*y | m] against [log lam | -lam]            (decoder.py:291-294);
      * dt_l [T] (naive Bayes) : A = [y | dt_t] against [ma log(tun+1e-20) | -sum ma tun], the row term
                                 gains -log(dt_t) sum_n ma y                        (decoder.py:73-85).
    The fp16 tensor-core kernel is used whenever A is exact in fp16 (integer counts <= 2048 and 0/1 masks);
    otherwise the fp32 CUDA-core tiles."""

    def __init__(self, y, ma_neuron=None, dt_l=None, impl=0, ones_col=False):
        _f32(y, "y", 2)
        self.T, self.N = y.shape
        self.mode = 0
        self.ma_vec = None
        self.per_bin_dt = dt_l is not None
        if ma_neuron is not None and ma_neuron.dim() == 2:
            self.mode = 1
            if dt_l is None:
                self.A = torch.cat([y * ma_neuron, ma_neuron], dim=1).contiguous()
                self.lgam = lgamma_rowsum(y, ma_neuron)
            else:
                # both options: A = [m*y | dt_t*m] against [log(tun+1e-20) | -(tun+1e-20)] (mode-1 operand at dt=1)
                self.A = torch.cat([y * ma_neuron, ma_neuron * dt_l.reshape(-1, 1)], dim=1).contiguous()
                lgam, ysum = lgamma_rowsum(y, ma_neuron, want_ysum=True)
                self.lgam = lgam - torch.log(dt_l) * ysum
        elif dt_l is not None:
            self.mode = 2
            self.ma_vec = ma_neuron
            self.A = torch.cat([y, dt_l.reshape(-1, 1)], dim=1).contiguous()
            lgam, ysum = lgamma_rowsum(y, ma_neuron, want_ysum=True)
            self.lgam = lgam - torch.log(dt_l) * ysum
        else:
            self.ma_vec = ma_neuron
            self.A = y
            if impl == 0:
                # one pass over the counts: fp16 copy, exactness flag and the lgamma row term
                self.A16 = CountsF16(y, ones_col=ones_col, ma_vec=ma_neuron, want_lgam=True)
                self.lgam = self.A16.lgam
                return
            self.lgam = lgamma_rowsum(y, ma_neuron)
        # per-bin dt is not fp16-exact: that path always runs on the fp32 tiles
        self.A16 = (CountsF16(self.A, ones_col=(ones_col and self.mode == 0))
                    if (impl == 0 and not self.per_bin_dt) else None)

    @property
    def tensor_cores(self):
        return self.A16 is not None and self.A16.exact

    def loglik(self, tuning, ma_latent=None, dt=1.0, out=None):
        """ll[T,K] for this recording under `tuning` [K,N]."""
        K = tuning.shape[0]
        if self.per_bin_dt:
            dt = 1.0                      # dt_t lives in the left-hand operand and the row term
        if self.mode == 0:
            return emission(self.A, tuning, self.lgam, self.ma_vec, ma_latent, dt, out=out, y16=self.A16,
                            impl=0 if self.tensor_cores else 1)
        if self.tensor_cores:
            bn = emission_tile_n(K)
            Kpad = (K + bn - 1) // bn * bn
            B, lam_sum = emission_prepare_aug(tuning, self.mode, self.ma_vec, dt, rows_out=Kpad)
            L16 = split_f16(B, out=torch.empty((2, Kpad, self.A16.ld), dtype=torch.float16, device=B.device))
            return emission_poisson_f16(self.A16, L16, lam_sum, self.lgam, K, ma_latent, out=out)
        B, lam_sum = emission_prepare_aug(tuning, self.mode, self.ma_vec, dt)
        return emission_poisson(self.A, B, lam_sum, self.lgam, ma_latent, out=out)


class GaussianEmission:
    """Emission operand of the Gaussian families (reference decoder.py:50-57): same interface as EmissionOperands.
    The observations are real-valued, so there is no fp16 copy (statistics and scans use the fp32 kernels)."""
    mode = 0
    A16 = None
    tensor_cores = False

    def __init__(self, y, ma_neuron=None, noise_std=0.5, impl=0, ones_col=False, dt_l=None):
        _f32(y, "y", 2)
        if dt_l is not None:
            raise ValueError("per-bin dt is a Poisson option (reference decoder.py:73-85)")
        self.y, self.ma, self.noise_std = y, ma_neuron, float(noise_std)
        self.T, self.N = y.shape
        if ma_neuron is not None:
            _f32(ma_neuron, "ma_neuron")
            if tuple(ma_neuron.shape) not in ((self.N,), (self.T, self.N)):
                raise ValueError("ma_neuron must be [N] or [T,N]")

    def loglik(self, tuning, ma_latent=None, dt=1.0, out=None):
        lib = _lib.load()
        _f32(tuning, "tuning", 2)
        K = tuning.shape[0]
        mu = tuning if dt == 1.0 else tuning * float(dt)
        if out is None:
            out = torch.empty((self.T, K), dtype=torch.float32, device=self.y.device)
        ldm = self.N if (self.ma is not None and self.ma.dim() == 2) else 0
        check(lib.pmg_emission_gaussian(self.T, self.N, K, _p(self.y), self.y.stride(0), _p(mu), _p(self.ma), ldm,
                                        self.noise_std, _p(ma_latent), _p(out), out.stride(0), _stream()),
              "pmg_emission_gaussian")
        _count(1)
        return out


def naive_bayes_normalize(ll, inplace=False, want_post=False):
    """(log_post[T,K], lml_t[T]) (reference decoder.py:98-101); want_post: also exp(log_post), in the same pass."""
    lib = _lib.load()
    _f32(ll, "ll", 2)
    T, K = ll.shape
    log_post = ll if inplace else torch.empty_like(ll)
    lml = torch.empty(T, dtype=torch.float32, device=ll.device)
    if want_post:
        post = torch.empty_like(ll)
        check(lib.pmg_naive_bayes_posterior(T, K, _p(ll), K, _p(log_post), _p(post), K, _p(lml), _stream()),
              "pmg_naive_bayes_posterior")
        _count(1)
        return log_post, lml, post
    check(lib.pmg_naive_bayes_normalize(T, K, _p(ll), K, _p(log_post), K, _p(lml), _stream()),
          "pmg_naive_bayes_normalize")
    _count(1)
    return log_post, lml


def naive_bayes_lml(ll, out=None):
    """lml_t[T] = logsumexp_k ll[t,:] alone (no log_post write), bit-identical to naive_bayes_normalize's lml_t."""
    lib = _lib.load()
    _f32(ll, "ll", 2)
    T, K = ll.shape
    if out is None:
        out = torch.empty(T, dtype=torch.float32, device=ll.device)
    elif out.dtype != torch.float32 or out.numel() != T or not out.is_contiguous():
        raise ValueError("out must be a contiguous float32 tensor of %d entries" % T)
    check(lib.pmg_naive_bayes_lml(T, K, _p(ll), ll.stride(0), _p(out), _stream()), "pmg_naive_bayes_lml")
    _count(1)
    return out


# ----------------------------------------------------------------------------- transitions
def stationary_joint(P0, M):
    """Stationary distribution pi[2,K] of T[(d,x),(d',x')] = M[d,d'] P_{d'}[x,x'] with P_1 = 1/K.
    The jump component is uniform, pi_1 = pi_d(1)/K; the move component solves
    pi_0 (I - M00 P0) = M10 pi_1 P0."""
    K = P0.shape[0]
    M = np.asarray(M, dtype=np.float64)
    pmj, pjm = M[0, 1], M[1, 0]
    if pmj + pjm <= 0:
        return np.full((2, K), 0.5 / K, dtype=np.float32)
    pd1 = pmj / (pmj + pjm)
    pi1 = np.full(K, pd1 / K)
    rhs = M[1, 0] * (pi1 @ P0)
    A = np.eye(K) - M[0, 0] * P0
    try:
        pi0 = np.linalg.solve(A.T, rhs)
    except np.linalg.LinAlgError:
        return np.full((2, K), 0.5 / K, dtype=np.float32)
    pi = np.stack([np.maximum(pi0, 0), pi1])
    return (pi / pi.sum()).astype(np.float32)


def dense_scan_pays(K, W):
    """The lockstep tensor-core scan costs ~3 K^2 tensor flops per bin and pass, a band kernel K (2W+1) CUDA-core
    flops: the GEMM form wins once the band covers a good part of the matrix."""
    return 256 <= K <= 4096 and (2 * W + 1) * 4 >= K        # (16 column tiles of 256: the kernel's limit)


class DenseMoveTC:
    """Right-hand operands of the lockstep scan GEMMs: the row-normalised move matrix P0 scaled by 2^14 as two fp16
    pieces, once transposed (forward pass: D[c,x'] = sum_x u[c,x] P0[x,x']) and once as is (backward pass), plus
    the 64-column block range every column tile touches (band structure)."""
    SCALE = 16384.0

    def __init__(self, P0, device):
        lib = _lib.load()
        P0 = np.asarray(P0, dtype=np.float64)
        K = P0.shape[0]
        geo = [C.c_int(0) for _ in range(4)]
        check(lib.pmg_dense_scan_geometry(K, *[C.byref(g) for g in geo]), "pmg_dense_scan_geometry")
        self.K, (self.Kk, self.Kn, self.BN, self.n_ntiles) = K, [g.value for g in geo]
        buf = np.zeros((2, 2, self.Kn, self.Kk), dtype=np.float16)
        rng = np.zeros((2, self.n_ntiles, 2), dtype=np.int32)
        for d, B in enumerate((P0.T, P0)):
            sc = B * self.SCALE
            hi = sc.astype(np.float16)
            lo = (sc - hi.astype(np.float64)).astype(np.float16)
            buf[d, 0, :K, :K] = hi
            buf[d, 1, :K, :K] = lo
            nz = (buf[d, 0] != 0) | (buf[d, 1] != 0)
            for i in range(self.n_ntiles):
                cols = np.nonzero(nz[i * self.BN:(i + 1) * self.BN].any(axis=0))[0]
                rng[d, i] = (cols.min() // 64, cols.max() // 64 + 1) if cols.size else (0, 1)
        self.P16 = torch.from_numpy(buf).to(device)
        self.kb_host = np.ascontiguousarray(rng)
        self.kb_ptr = self.kb_host.ctypes.data_as(C.POINTER(C.c_int))
        self._ws = {}

    def workspace(self, n_chain, device):
        ws = self._ws.get(n_chain)
        if ws is None:
            nbytes = int(_lib.load().pmg_dense_scan_workspace_bytes(int(n_chain), self.K))
            ws = self._ws[n_chain] = torch.empty(nbytes, dtype=torch.uint8, device=device)
        return ws

    def chains(self, sm_count):
        """chains that fill the GPU with one wave of 128-chain x BN-column accumulator tiles"""
        return 128 * max(1, sm_count // self.n_ntiles)


class MoveOperator:
    """Device copy of the factored "move" transition + the 2x2 dynamics matrix."""

    def __init__(self, host, M, device, P0=None, dense_tc=None):
        """P0: optional dense row-normalised move matrix [K,K] (host); when given, the stationary
        distribution of the joint (dynamics x latent) prior chain is computed and used as the
        message that time-parallel warm-ups start from.
        dense_tc: run mode-0 passes as lockstep tensor-core GEMMs (None = when the band is wide enough to pay)."""
        self.K = int(host["inv_z"].shape[0]) if host["kind"] == 0 else int(host["band_fwd"].shape[1])
        self.kind, self.W = int(host["kind"]), int(host["W"])
        self.M = np.asarray(M, dtype=np.float32).reshape(4)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        self.taps = dev(host["taps"]) if self.kind == 0 else None
        self.inv_z = dev(host["inv_z"]) if self.kind == 0 else None
        self.band_fwd = dev(host["band_fwd"]) if self.kind == 1 else None
        self.band_bwd = dev(host["band_bwd"]) if self.kind == 1 else None
        self.stationary = None
        if P0 is not None:
            self.stationary = dev(stationary_joint(np.asarray(P0, dtype=np.float64), self.M.reshape(2, 2)))
        # dense / wide-band kernels: lockstep tensor-core scan (pmg_forward_dense / pmg_backward_dense)
        self.dense = None
        if dense_tc is None:
            dense_tc = P0 is not None and dense_scan_pays(self.K, self.W)
        if dense_tc:
            if P0 is None:
                raise ValueError("the tensor-core scan needs the dense row-normalised move matrix P0")
            self.dense = DenseMoveTC(P0, device)

    def cstruct(self):
        """ctypes view of the operator (built once: the device arrays never move)"""
        s = getattr(self, "_cs", None)
        if s is not None:
            return s
        s = self._cs = PmgTransition()
        s.K, s.kind, s.W = self.K, self.kind, self.W
        s.taps = self.taps.data_ptr() if self.taps is not None else None
        s.inv_z = self.inv_z.data_ptr() if self.inv_z is not None else None
        s.band_fwd = self.band_fwd.data_ptr() if self.band_fwd is not None else None
        s.band_bwd = self.band_bwd.data_ptr() if self.band_bwd is not None else None
        for i in range(4):
            s.M[i] = float(self.M[i])
        return s


def make_plan(T, core_begin, core_end, chunk_len, halo, left_exact, right_exact, likelihood_scale, halo_next=0):
    p = PmgScanPlan()
    p.T, p.core_begin, p.core_end = int(T), int(core_begin), int(core_end)
    p.chunk_len = int(chunk_len)
    p.n_chain = int((core_end - core_begin + chunk_len - 1) // chunk_len)
    p.halo = int(halo)
    p.left_exact, p.right_exact = int(bool(left_exact)), int(bool(right_exact))
    p.likelihood_scale = float(likelihood_scale)
    p.halo_next = int(halo_next)
    p.sel_tol, p.sel_err = 0.0, None
    p.halo_arr = p.halo_next_arr = None
    return p


def set_chain_halos(plan, cur=None, nxt=None):
    """Per-chain warm-up lengths (device int32 [n_chain]) of this pass / the next pass, or None for the scalars."""
    for t in (cur, nxt):
        if t is not None and (t.dtype != torch.int32 or t.numel() < plan.n_chain or not t.is_contiguous()):
            raise ValueError("per-chain halos must be contiguous int32 [n_chain]")
    plan.halo_arr = cur.data_ptr() if cur is not None else None
    plan.halo_next_arr = nxt.data_ptr() if nxt is not None else None


def _select(plan, mode, sel_err, sel_tol):
    """mode 2: the chains to re-run are selected on the device, chain s iff !(sel_err[s] <= sel_tol)."""
    if mode == 2:
        if sel_err is None or sel_err.numel() < plan.n_chain:
            raise ValueError("mode 2 needs one seam error per chain")
        plan.sel_err, plan.sel_tol = sel_err.data_ptr(), float(sel_tol)
    else:
        plan.sel_err, plan.sel_tol = None, 0.0


def _warm(warm_in):
    """(pointer, stride): one [2,K] vector shared by all chains, or [n_chain,2,K] with one per chain."""
    if warm_in is None:
        return None, 0
    return _p(warm_in), (0 if warm_in.dim() == 2 else warm_in.stride(0))


def forward(plan, op, ll, alpha, lmr, halo_state=None, carry_in=None, mode=0, chain_ids=None, warm_in=None,
            warm_out=None, sel_err=None, sel_tol=0.0, halo_max=0):
    """halo_max: upper bound of the per-chain warm-ups set with set_chain_halos (lockstep scan only)."""
    lib = _lib.load()
    _select(plan, mode, sel_err, sel_tol)
    tr = op.cstruct()
    n_ids = int(chain_ids.numel()) if chain_ids is not None else 0
    wp, ws = _warm(warm_in)
    dense = getattr(op, "dense", None)
    if mode == 0 and dense is not None:
        wk = dense.workspace(plan.n_chain, ll.device)
        check(lib.pmg_forward_dense(C.byref(plan), C.byref(tr), _p(dense.P16), dense.kb_ptr, int(halo_max), _p(ll),
                                    ll.shape[1], _p(carry_in), wp, ws, _p(warm_out), _p(alpha), _p(lmr),
                                    _p(halo_state), _p(wk), wk.numel(), _stream()), "pmg_forward_dense")
        _count(2 * (max(plan.halo, int(halo_max)) + plan.chunk_len) + 1)
        return
    check(lib.pmg_forward(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(carry_in), wp, ws, _p(warm_out),
                          _p(alpha), _p(lmr),
                          _p(halo_state), int(mode), _p(chain_ids), n_ids, _stream()), "pmg_forward")
    _count(1)


def backward(plan, op, ll, alpha, gamma=None, gamma_lat=None, dyn_marg=None, r_out=None, tw_partial=None,
             beta_halo=None, beta_end=None, beta_in=None, mode=0, chain_ids=None, gamma16=None, warm_in=None,
             warm_out=None, sel_err=None, sel_tol=0.0, halo_max=0, xi16=None):
    """xi16: optional bf16 [4, T, 2K] (alpha hi, alpha lo, r hi, r lo) that receives the operands of the
    transition-count GEMM as pieces instead of ``r_out`` (see xi16_supported)."""
    lib = _lib.load()
    _select(plan, mode, sel_err, sel_tol)
    tr = op.cstruct()
    n_ids = int(chain_ids.numel()) if chain_ids is not None else 0
    wp, ws = _warm(warm_in)
    dense = getattr(op, "dense", None)
    if xi16 is not None:
        if r_out is not None or xi16.dtype != torch.bfloat16 or xi16.dim() != 3 or xi16.shape[0] != 4:
            raise ValueError("xi16 must be bfloat16 [4, T, 2K] and replaces r_out")
        check(lib.pmg_backward_xi16(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(alpha), _p(beta_in), wp, ws,
                                    _p(warm_out), _p(gamma), _p(gamma_lat), _p(gamma16),
                                    (gamma16.shape[2] if gamma16 is not None else 0), _p(dyn_marg), _p(xi16[0]),
                                    _p(xi16[1]), _p(xi16[2]), _p(xi16[3]), xi16.shape[2], _p(tw_partial),
                                    _p(beta_halo), _p(beta_end), int(mode), _p(chain_ids), n_ids, _stream()),
              "pmg_backward_xi16")
        _count(1)
        return
    if mode == 0 and dense is not None:
        wk = dense.workspace(plan.n_chain, ll.device)
        check(lib.pmg_backward_dense(C.byref(plan), C.byref(tr), _p(dense.P16), dense.kb_ptr, int(halo_max), _p(ll),
                                     ll.shape[1], _p(alpha), _p(beta_in), wp, ws, _p(warm_out), _p(gamma),
                                     _p(gamma_lat), _p(gamma16), (gamma16.shape[2] if gamma16 is not None else 0),
                                     _p(dyn_marg), _p(r_out), _p(tw_partial), _p(beta_halo), _p(beta_end), _p(wk),
                                     wk.numel(), _stream()), "pmg_backward_dense")
        _count(2 * (max(plan.halo, int(halo_max)) + plan.chunk_len))
        return
    check(lib.pmg_backward(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(alpha), _p(beta_in), wp, ws,
                           _p(warm_out), _p(gamma),
                           _p(gamma_lat), _p(gamma16), (gamma16.shape[2] if gamma16 is not None else 0), _p(dyn_marg),
                           _p(r_out), _p(tw_partial), _p(beta_halo), _p(beta_end),
                           int(mode), _p(chain_ids), n_ids, _stream()), "pmg_backward")
    _count(1)


def viterbi_bp(T, K, device):
    """int16 [T, 2, ldbp] backpointer buffer of viterbi_forward (ldbp = K rounded up to 8; rows need no init)."""
    return torch.empty((T, 2, (K + 7) // 8 * 8), dtype=torch.int16, device=device)


def viterbi_forward(plan, op, ll, bp, lmr, halo_state=None, end_msg=None, carry_in=None, mode=0, chain_ids=None,
                    warm_in=None, warm_out=None, sel_err=None, sel_tol=0.0):
    """Max-product forward pass with backpointers (pmg_viterbi_forward): pmg_forward's plan, warm-start and repair
    conventions; bp from viterbi_bp, end_msg [n_chain,2,K] = message at each chain's last core bin."""
    lib = _lib.load()
    if bp.dtype != torch.int16 or bp.dim() != 3 or bp.shape[1] != 2 or not bp.is_contiguous():
        raise ValueError("bp must be a contiguous int16 [T, 2, ldbp] tensor")
    _select(plan, mode, sel_err, sel_tol)
    tr = op.cstruct()
    n_ids = int(chain_ids.numel()) if chain_ids is not None else 0
    wp, ws = _warm(warm_in)
    check(lib.pmg_viterbi_forward(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(carry_in), wp, ws,
                                  _p(warm_out), _p(bp), bp.shape[2], _p(lmr), _p(halo_state), _p(end_msg), int(mode),
                                  _p(chain_ids), n_ids, _stream()), "pmg_viterbi_forward")
    _count(1)


def viterbi_chain_maps(plan, K, bp, maps):
    """maps [n_chain, 2K] int32: state at each chain's first core bin on the best path ending in each state."""
    check(_lib.load().pmg_viterbi_chain_maps(C.byref(plan), int(K), _p(bp), bp.shape[2], _p(maps), _stream()),
          "pmg_viterbi_chain_maps")
    _count(1)


def viterbi_backtrack(plan, K, bp, maps, last_msg, path):
    """path [T] int32 (core bins) = flat states d*K + x of the MAP path ending in argmax(last_msg)."""
    check(_lib.load().pmg_viterbi_backtrack(C.byref(plan), int(K), _p(bp), bp.shape[2], _p(maps), _p(last_msg),
                                            _p(path), _stream()), "pmg_viterbi_backtrack")
    _count(2)


def viterbi_records(n, K, device):
    """n zeroed records of a time-sharded Viterbi backtrack, int32 [n, 4K + 2] in the layout
    pmg_viterbi_backtrack_sharded reads: link [2K] int32 | last message [2K] fp32 | partial sum of lmr (fp64)."""
    return torch.zeros((n, 4 * K + 2), dtype=torch.int32, device=device)


def split_viterbi_records(gathered, K):
    """[n, 4K + 2] int32 records -> (link [n, 2K] int32, msg [n, 2K] fp32, lsum [n] fp64) views."""
    return (gathered[:, :2 * K], gathered[:, 2 * K:4 * K].view(torch.float32),
            gathered[:, 4 * K:].view(torch.float64).view(-1))


def viterbi_block_link(plan, K, bp, maps, link):
    """link [2K] int32: state at bin core_begin - 1 on the best path ending in each state at core_end - 1."""
    check(_lib.load().pmg_viterbi_block_link(C.byref(plan), int(K), _p(bp), bp.shape[2], _p(maps), _p(link),
                                             _stream()), "pmg_viterbi_block_link")
    _count(1)


def viterbi_backtrack_sharded(plan, K, bp, maps, gathered, rank, path):
    """path [T] int32 (core bins) of this rank's block of the MAP path; gathered [world, 4K + 2] int32 records."""
    if gathered.dtype != torch.int32 or gathered.dim() != 2 or gathered.shape[1] != 4 * K + 2 \
            or not gathered.is_contiguous():
        raise ValueError("gathered must be contiguous int32 [world, 4K + 2]")
    check(_lib.load().pmg_viterbi_backtrack_sharded(C.byref(plan), int(K), _p(bp), bp.shape[2], _p(maps),
                                                    _p(gathered), gathered.shape[0], int(rank), _p(path), _stream()),
          "pmg_viterbi_backtrack_sharded")
    _count(2)


def scan_compact_supported(op, likelihood_scale):
    """True when the EM fast path (pmg_forward_compact / pmg_backward_compact) covers this transition."""
    tr = op.cstruct()
    return bool(_lib.load().pmg_scan_compact_supported(C.byref(tr), float(likelihood_scale)))


def forward_compact(plan, op, ll, ax, halo_state=None, fwd_end=None, first_out=None, carry_in=None, mode=0,
                    chain_ids=None, warm_in=None, warm_out=None, sel_err=None, sel_tol=0.0):
    """Forward pass writing the compact filtered posterior ax [T, K+4] (alpha[0,:], a1s, lmr per bin)."""
    lib = _lib.load()
    _select(plan, mode, sel_err, sel_tol)
    tr = op.cstruct()
    n_ids = int(chain_ids.numel()) if chain_ids is not None else 0
    wp, ws = _warm(warm_in)
    check(lib.pmg_forward_compact(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(carry_in), wp, ws,
                                  _p(warm_out), _p(ax), ax.shape[1], _p(halo_state), _p(fwd_end), _p(first_out),
                                  int(mode), _p(chain_ids), n_ids, _stream()), "pmg_forward_compact")
    _count(1)


def backward_compact(plan, op, ll, ax, gamma16, beta_halo=None, beta_end=None, beta_in=None,
                     mode=0, chain_ids=None, warm_in=None, warm_out=None, sel_err=None, sel_tol=0.0):
    """Backward pass of an EM iteration: fp16 pieces of the latent posterior (and the seam messages)."""
    lib = _lib.load()
    _select(plan, mode, sel_err, sel_tol)
    tr = op.cstruct()
    n_ids = int(chain_ids.numel()) if chain_ids is not None else 0
    wp, ws = _warm(warm_in)
    check(lib.pmg_backward_compact(C.byref(plan), C.byref(tr), _p(ll), ll.shape[1], _p(ax), ax.shape[1],
                                   _p(beta_in), wp, ws, _p(warm_out), _p(gamma16), gamma16.shape[2],
                                   _p(beta_halo), _p(beta_end), int(mode), _p(chain_ids), n_ids,
                                   _stream()), "pmg_backward_compact")
    _count(1)


def boundary_pack_fwd(K, out, first, last, warm_src=None, ax_row=None, ll_row=None, scale=1.0):
    """out [8K] <- [first | 0 | last | warm]; warm = warm_src [2K], or the compact row (ax_row, ll_row), or zeros."""
    mode = 2 if ax_row is not None else (1 if warm_src is not None else 0)
    check(_lib.load().pmg_boundary_pack_fwd(int(K), _p(first), _p(last), mode, _p(warm_src), _p(ax_row), _p(ll_row),
                                            float(scale), _p(out), _stream()), "pmg_boundary_pack_fwd")
    _count(1)


def boundary_unpack_fwd(K, from_left, from_right, fwd_end0, fwarm0, ax_stop=None, ll_stop=None, scale=1.0,
                        alpha_stop=None):
    """from_left [4K] -> fwd_end0, fwarm0; from_right [4K] -> the row behind the block (compact: ax_stop + ll_stop)."""
    if from_left is None and from_right is None:
        return
    check(_lib.load().pmg_boundary_unpack_fwd(int(K), _p(from_left), _p(from_right), _p(fwd_end0), _p(fwarm0),
                                              int(ax_stop is not None), _p(ax_stop), _p(ll_stop), float(scale),
                                              _p(alpha_stop), _stream()), "pmg_boundary_unpack_fwd")
    _count(1)


def seam_check(n, length, est_ptr, ld_est, truth_ptr, ld_truth, err, floor_val=1e-12):
    """err[i] = max relative difference of the unit-sum-normalised messages over entries > floor_val.  Entries
    below 1e-12 of a normalised message cannot reach 1e-7 in any posterior (every state is entered by a jump with
    probability >= p_move_to_jump/K per bin, which bounds the ratio of backward-message entries)."""
    lib = _lib.load()
    check(lib.pmg_seam_check(int(n), int(length), C.c_void_p(est_ptr), int(ld_est), C.c_void_p(truth_ptr),
                             int(ld_truth), float(floor_val), _p(err), _stream()), "pmg_seam_check")
    _count(1)


def seam_check_fix(n, length, est_ptr, ld_est, truth_ptr, ld_truth, err, tol, fix=False, counter=None,
                   floor_val=1e-12):
    """seam_check that also counts the seams with !(err <= tol) into `counter` (one device float) and, with fix=True,
    overwrites their estimate by the truth: the snapshot a mode-2 restart of that chain starts from."""
    lib = _lib.load()
    check(lib.pmg_seam_check_fix(int(n), int(length), C.c_void_p(est_ptr), int(ld_est), C.c_void_p(truth_ptr),
                                 int(ld_truth), float(floor_val), float(tol), int(bool(fix)), _p(err), _p(counter),
                                 _stream()), "pmg_seam_check_fix")
    _count(1)


# ----------------------------------------------------------------------------- reductions over time
def strided_sum_workspace(device):
    """zero-initialised scratch of pmg_strided_sum (one per caller: calls sharing it must be stream-ordered)"""
    n = int(_lib.load().pmg_strided_sum_workspace_bytes())
    return torch.zeros((n + 7) // 8, dtype=torch.int64, device=device)


def strided_sum(src, dst, ws):
    """dst[0] = sum(src) for a 1-D float32 view `src` (any stride), fp64 accumulation, one launch."""
    if src.dim() != 1 or src.dtype != torch.float32 or dst.dtype != torch.float32:
        raise TypeError("strided_sum expects a 1-D float32 view and a float32 destination")
    check(_lib.load().pmg_strided_sum(int(src.shape[0]), _p(src), int(src.stride(0)) if src.shape[0] > 1 else 1, _p(dst),
                                      _p(ws), _stream()), "pmg_strided_sum")
    _count(1)


_ws_cache = {}


def _workspace(nbytes, device):
    key = (device.index if device.index is not None else torch.cuda.current_device())
    ws = _ws_cache.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = ws
    return ws


def atb(A, B, out=None, impl=0):
    """C[M,N] = sum_t A[t,:M]^T B[t,:N].  A and B may be row-offset views of 2-D tensors."""
    lib = _lib.load()
    if A.dim() != 2 or B.dim() != 2 or A.shape[0] != B.shape[0]:
        raise ValueError("atb expects [T,M] and [T,N]")
    for t, nm in ((A, "A"), (B, "B")):
        if t.dtype != torch.float32 or not t.is_cuda or t.stride(1) != 1:
            raise TypeError("%s must be a float32 CUDA tensor with unit inner stride" % nm)
    T, M = A.shape
    N = B.shape[1]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    nbytes = lib.pmg_atb_workspace_bytes(T, M, N, int(impl))
    ws = _workspace(nbytes, A.device)
    check(lib.pmg_atb(T, M, N, _p(A), A.stride(0), _p(B), B.stride(0), _p(out), out.stride(0), _p(ws), ws.numel(), int(impl),
                      _stream()), "pmg_atb")
    _count(2)
    return out


def new_gamma16(T, K, device):
    """[2, T, ldg] fp16 buffer for the hi/lo pieces of the posterior (padding columns zero)."""
    ldg = (K + 7) // 8 * 8
    return torch.zeros((2, T, ldg), dtype=torch.float16, device=device)


def split_f16(src, out=None):
    """fp32 [T,K] -> fp16 hi/lo pieces [2,T,ldg]."""
    lib = _lib.load()
    _f32(src, "src", 2)
    T, K = src.shape
    if out is None:
        out = new_gamma16(T, K, src.device)
    check(lib.pmg_split_f16(T, K, _p(src), K, _p(out), out.shape[2], _stream()), "pmg_split_f16")
    _count(1)
    return out


def atb_f16(g16, y16, K, out=None):
    """yw[K,N] = sum_t gamma[t,:K]^T y[t,:N] on the tensor cores (fp16 pieces, fp32 accumulation).
    With a ones column in y16 the result is [K, N+1] and its last column is sum_t gamma."""
    lib = _lib.load()
    T, N = y16.T, y16.N + (1 if y16.ones_col else 0)
    if g16.shape[1] != T:
        raise ValueError("posterior pieces have %d bins, counts have %d" % (g16.shape[1], T))
    if out is None:
        out = torch.empty((K, N), dtype=torch.float32, device=g16.device)
    nbytes = lib.pmg_atb_f16_workspace_bytes(T, K, N)
    ws = _workspace(nbytes, g16.device)
    check(lib.pmg_atb_f16(T, K, N, _p(g16), g16.shape[2], _p(y16.data), y16.ld, _p(out), _p(ws), ws.numel(),
                          _stream()), "pmg_atb_f16")
    _count(2)
    return out


def split_bf16(src):
    """fp32 [T,K] (row stride >= K) -> bf16 hi/lo pieces [2,T,ld], ld = K rounded up to 8."""
    lib = _lib.load()
    if src.dim() != 2 or src.dtype != torch.float32 or not src.is_cuda or src.stride(1) != 1:
        raise TypeError("split_bf16 expects a float32 CUDA matrix with unit inner stride")
    T, K = src.shape
    ld = (K + 7) // 8 * 8
    out = (torch.zeros if ld != K else torch.empty)((2, T, ld), dtype=torch.bfloat16, device=src.device)
    check(lib.pmg_split_bf16(T, K, _p(src), src.stride(0), _p(out), ld, _stream()), "pmg_split_bf16")
    _count(1)
    return out


XI_TC_MIN_BINS = 4096        # shorter recordings: the fp32 CUDA-core reduction (no piece rounding) is as fast


def atb_bf16x2(A, B, out=None):
    """C[M,N] = sum_t A[t,:M]^T B[t,:N] on the tensor cores: both operands as two bf16 pieces, three products
    (relative error ~2^-16 per term, fp32 accumulation).  The transition-count GEMM of decode_latent."""
    lib = _lib.load()
    if A.dim() != 2 or B.dim() != 2 or A.shape[0] != B.shape[0]:
        raise ValueError("atb expects [T,M] and [T,N]")
    T, M = A.shape
    N = B.shape[1]
    a16, b16 = split_bf16(A), split_bf16(B)
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=A.device)
    nbytes = lib.pmg_atb_f16_workspace_bytes(T, M, N)
    ws = _workspace(nbytes, A.device)
    check(lib.pmg_atb_bf16x2(T, M, N, _p(a16), a16.shape[2], _p(b16), b16.shape[2], _p(out), _p(ws), ws.numel(),
                             _stream()), "pmg_atb_bf16x2")
    _count(2)
    return out


def xi16_supported(op, likelihood_scale):
    """True when the backward pass can write the transition-count operands as bf16 pieces itself (bulk kernel)."""
    if getattr(op, "dense", None) is not None:
        return False
    tr = op.cstruct()
    return bool(_lib.load().pmg_backward_xi16_supported(C.byref(tr), float(likelihood_scale)))


def atb_bf16x2_pieces(xi16, row0, n_rows, M=None, N=None, out=None):
    """sum_t alpha_t^T (r_{t+1} / z_t) over the pairs t in [row0, row0 + n_rows) from the pieces of
    backward(..., xi16=...): alpha rows [row0, row0+n) against r rows [row0+1, row0+n+1).  M, N: leading columns used
    of the two operands (default all 2K; the latent-only families use the first K)."""
    lib = _lib.load()
    ld = xi16.shape[2]
    M = ld if M is None else int(M)
    N = ld if N is None else int(N)
    T = int(n_rows)
    a_hi, a_lo = xi16[0, row0:row0 + T], xi16[1, row0:row0 + T]
    r_hi, r_lo = xi16[2, row0 + 1:row0 + 1 + T], xi16[3, row0 + 1:row0 + 1 + T]
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=xi16.device)
    nbytes = lib.pmg_atb_f16_workspace_bytes(T, M, N)
    ws = _workspace(nbytes, xi16.device)
    # operand roles of pmg_atb_bf16x2: out[k, n] = sum_t G[t, k] Y[t, n] with G = alpha, Y = r
    check(lib.pmg_atb_bf16x2_pieces(T, M, N, _p(a_hi), _p(a_lo), ld, _p(r_hi), _p(r_lo), ld, _p(out), _p(ws),
                                    ws.numel(), _stream()), "pmg_atb_bf16x2_pieces")
    _count(2)
    return out


def xi_finalize(G, logP, logM_host):
    lib = _lib.load()
    _f32(G, "G", 2); _f32(logP, "logP", 3)
    K = logP.shape[1]
    out = torch.empty((2, 2, K, K), dtype=torch.float32, device=G.device)
    lm = (C.c_float * 4)(*[float(v) for v in np.asarray(logM_host, dtype=np.float32).reshape(4)])
    check(lib.pmg_xi_finalize(K, _p(G), _p(logP), lm, _p(out), _stream()), "pmg_xi_finalize")
    _count(1)
    return out


# ----------------------------------------------------------------------------- M-step
class AdamState:
    """optax.adam state (count, mu, nu) kept on the device across EM iterations
    (reference core.py:662, fit_tuning_helper.py:131-132)."""

    def __init__(self, params):
        self.count = torch.zeros(1, dtype=torch.int32, device=params.device)
        self.mu = torch.zeros_like(params)
        self.nu = torch.zeros_like(params)

    @classmethod
    def packed(cls, params):
        """State whose weights and moments are views of ONE buffer `flat` [3,B,N] = (W, mu, nu): a single copy
        snapshots or restores the optimiser (the EM loop does that once per iteration)."""
        st = cls.__new__(cls)
        st.flat = torch.zeros((3,) + tuple(params.shape), dtype=torch.float32, device=params.device)
        st.flat[0].copy_(params)
        st.W, st.mu, st.nu = st.flat[0], st.flat[1], st.flat[2]
        st.count = torch.zeros(1, dtype=torch.int32, device=params.device)
        return st


def mstep_adam(Phi, yw, tw, W, state, prior_std, step_size=0.01, maxiter=1000, tol=1e-6, min_iters=5,
               b1=0.9, b2=0.999, eps=1e-8, out=None):
    """Runs the whole Adam loop on the device.  W and state are updated in place.
    Returns device tensors (loss_hist[maxiter], err_hist[maxiter], n_iter[1] int32, final[2], tuning[K,N]);
    out: optional tuple of preallocated tensors of those shapes to write into."""
    lib = _lib.load()
    _f32(Phi, "Phi", 2); _f32(W, "W", 2)
    K, B = Phi.shape
    N = W.shape[1]
    # yw / tw may be strided views ([K, N+1] statistics of atb_f16 consumed in place)
    for t, nm in ((yw, "yw"), (tw, "tw")):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != torch.float32:
            raise TypeError("%s must be a float32 CUDA tensor" % nm)
    if W.shape[0] != B or tuple(yw.shape) != (K, N) or tuple(tw.shape) != (K,) or yw.stride(1) != 1:
        raise ValueError("inconsistent M-step shapes")
    dev = W.device
    maxiter = int(maxiter)
    if out is not None:
        loss_hist, err_hist, n_iter, final, tuning = out
        if (loss_hist.numel() != maxiter or err_hist.numel() != maxiter or n_iter.numel() != 1 or final.numel() != 2
                or tuple(tuning.shape) != (K, N) or n_iter.dtype != torch.int32
                or not all(t.is_contiguous() for t in out)):
            raise ValueError("mstep_adam: out buffers have the wrong shape")
        _f32(loss_hist, "loss_hist"); _f32(err_hist, "err_hist"); _f32(final, "final"); _f32(tuning, "tuning", 2)
    else:
        loss_hist = torch.empty(maxiter, dtype=torch.float32, device=dev)
        err_hist = torch.empty(maxiter, dtype=torch.float32, device=dev)
        n_iter = torch.empty(1, dtype=torch.int32, device=dev)
        final = torch.empty(2, dtype=torch.float32, device=dev)
        tuning = torch.empty((K, N), dtype=torch.float32, device=dev)
    nbytes = lib.pmg_mstep_workspace_bytes(K, B, N, maxiter)
    ws = _workspace(nbytes, dev)
    check(lib.pmg_mstep_adam_ld(K, B, N, _p(Phi), _p(yw), int(yw.stride(0)), _p(tw), int(tw.stride(0)),
                                float(prior_std), float(step_size), float(b1),
                                float(b2), float(eps), maxiter, float(tol), int(min_iters), _p(W), _p(state.mu),
                                _p(state.nu), _p(state.count), _p(loss_hist), _p(err_hist), _p(n_iter), _p(final),
                                _p(tuning), _p(ws), ws.numel(), _stream()), "pmg_mstep_adam")
    _count(1)
    return loss_hist, err_hist, n_iter, final, tuning


def tuning_softplus(Phi, W):
    """softplus(Phi @ W) (reference fit_tuning_helper.py:11-25)."""
    lib = _lib.load()
    _f32(Phi, "Phi", 2); _f32(W, "W", 2)
    K, B = Phi.shape
    N = W.shape[1]
    out = torch.empty((K, N), dtype=torch.float32, device=W.device)
    check(lib.pmg_tuning_softplus(K, B, N, _p(Phi), _p(W), _p(out), _stream()), "pmg_tuning_softplus")
    _count(1)
    return out


# ----------------------------------------------------------------------------- initial posterior (jax bit stream)
def threefry_posterior_init(T, K, key, random_scale, device, t_offset=0, T_total=None, want_post=False,
                            want_log=False, g16=None, g16_row0=0, want_tw=False):
    """Rows [t_offset, t_offset+T) of the reference's initial posterior (core.py:571-583) generated on the
    device with jax.random's threefry stream.  g16: optional [2, T_ext, ldg] fp16 piece buffer; rows
    g16_row0 .. g16_row0+T-1 receive the hi/lo pieces.  Returns (post | None, logpost | None, tw fp32 | None)."""
    from . import jaxprng
    lib = _lib.load()
    k = jaxprng.as_key(key)
    T_total = int(T if T_total is None else T_total)
    f32 = dict(dtype=torch.float32, device=device)
    post = torch.empty((T, K), **f32) if want_post else None
    logp = torch.empty((T, K), **f32) if want_log else None
    tw = torch.empty(K, dtype=torch.float64, device=device) if want_tw else None
    gptr, ldg, stride = None, 0, 0
    if g16 is not None:
        ldg = g16.shape[2]
        stride = g16.shape[1] * ldg
        gptr = C.c_void_p(g16.data_ptr() + int(g16_row0) * ldg * 2)
    check(lib.pmg_threefry_posterior_init(int(T), int(K), int(t_offset), T_total, int(k[0]), int(k[1]),
                                          float(random_scale), _p(post), K, _p(logp), K, gptr, ldg, stride,
                                          _p(tw), _stream()), "pmg_threefry_posterior_init")
    _count(1)
    return post, logp, (tw.to(torch.float32) if tw is not None else None)
