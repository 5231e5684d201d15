"""CPU-only tests: C-ABI surface, host-side logic, product/oracle separation."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import ref_numpy as ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from poor_man_gplvm_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(libpath):
    hdr = open(os.path.join(ROOT, "include", "pmgplvm_b200.h")).read()
    declared = set(re.findall(r"\b(pmg_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 15
    lib = ctypes.CDLL(libpath)
    for name in declared:
        assert hasattr(lib, name), name
    from poor_man_gplvm_b200 import _lib
    assert set(_lib.SIGNATURES) == declared
    lib2 = _lib.load()
    assert lib2.pmg_version() >= 100
    assert lib2.pmg_error_string(-1) == b"bad argument"


def test_struct_layouts_match_header():
    from poor_man_gplvm_b200._lib import PmgScanPlan, PmgTransition
    # int K,kind,W (+4 pad) ; 4 pointers ; float[4]
    assert ctypes.sizeof(PmgTransition) == 16 + 32 + 16
    # 4 x int64 ; 4 x int ; float likelihood_scale, int halo_next, float sel_tol (+4 pad) ; pointer sel_err
    assert ctypes.sizeof(PmgScanPlan) == 32 + 16 + 16 + 3 * 8
    assert PmgScanPlan.sel_err.offset == 64 and PmgScanPlan.halo_next.offset == 52


def test_transition_and_basis_match_oracle():
    from poor_man_gplvm_b200 import gp_kernel as gpk
    for K, mv in ((50, 1.0), (100, 2.5)):
        P, logP, M, logM = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), mv, 0.02, 0.03)
        Po, logPo, Mo, logMo = ref.create_transition_prob_1d(K, mv, 0.02, 0.03, dtype=np.float32)
        assert np.allclose(P, Po, atol=1e-7) and np.allclose(logP, logPo, atol=1e-5)
        assert np.allclose(M, Mo) and np.allclose(logM, logMo)
    B = gpk.generate_basis(10.0, 100)
    Bo = ref.generate_basis(10.0, 100, dtype=np.float32)
    assert B.shape == Bo.shape == (100, 18)                       # SURVEY §8(a): B=18 at K=100, ls=10
    assert np.allclose(np.abs(B), np.abs(Bo), atol=1e-4)          # SVD sign ambiguity (SURVEY H6)


@pytest.mark.parametrize("K,mv", [(40, 1.0), (64, 3.0)])
def test_move_operator_factorisation_reconstructs_P0(K, mv):
    from poor_man_gplvm_b200 import gp_kernel as gpk
    P, *_ = gpk.create_transition_prob_1d(np.arange(K), np.arange(2), mv)
    h = gpk.move_operator_host(K, mv)
    assert h["kind"] == 0 and h["W"] <= int(10.2 * mv)
    x = np.arange(K)
    d = np.abs(x[:, None] - x[None, :])
    rec = np.where(d <= h["W"], h["taps"][np.minimum(d, h["W"])], 0) * h["inv_z"][:, None]
    assert np.max(np.abs(rec - P[0])) < 1e-7
    rng = np.random.default_rng(0)
    ck = rng.random((K, K)) * (d <= 5)
    ck[np.arange(K), np.arange(K)] += 0.1
    h = gpk.move_operator_host(K, mv, ck)
    P0 = ck / ck.sum(axis=1, keepdims=True)
    assert h["kind"] == 1 and h["W"] == 5
    W = h["W"]
    for j in range(2 * W + 1):
        for xx in range(K):
            src = xx - W + j
            if 0 <= src < K:
                assert np.isclose(h["band_fwd"][j, xx], P0[src, xx])
                assert np.isclose(h["band_bwd"][j, xx], P0[xx, src])


def test_plan_chunks_bounds():
    from poor_man_gplvm_b200.estep import plan_chunks, MIN_CHUNK
    assert plan_chunks(400, 256, 148) == 400                      # short sequences: one exact chain
    c = plan_chunks(10 ** 6, 256, 148)
    assert c >= 2 * 256 and (10 ** 6 + c - 1) // c <= 148 * 8
    assert (10 ** 6 + c - 1) // c > 148 * 7                       # the headline run fills every SM
    c12 = plan_chunks(10 ** 6, 256, 148, 12)                      # EM-mode plan of the compact kernels
    assert c12 >= 2 * 256 and 148 * 11 < (10 ** 6 + c12 - 1) // c12 <= 148 * 12
    assert plan_chunks(5000, 0, 148) == 5000
    # one-shot passes keep chunks of at least two warm-ups; EM mode (adaptive warm-up) fills the chain slots even
    # for a rank's share of a time-sharded recording (T = 1e6 over 8 ranks)
    assert plan_chunks(125000, 256, 148, 12) == 512
    assert plan_chunks(125000, 256, 148, 12, min_chunk=MIN_CHUNK) == 71


def test_model_constructs_on_cpu_and_fails_loudly_without_gpu():
    import torch
    import poor_man_gplvm_b200 as pmg
    m = pmg.PoissonGPLVMJump1D(8, 20, tuning_lengthscale=4.0)
    assert m.tuning.shape == (20, 8) and m.params.shape == (m.n_basis, 8)
    assert np.all(m.tuning > 0) and m.tuning_basis[:, 0].tolist() == [1.0] * 20
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            m.decode_latent_naive_bayes(np.zeros((5, 8), np.float32))


def test_product_sources_never_touch_the_oracle():
    pkg = os.path.join(ROOT, "poor_man_gplvm_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "/root/reference" not in src, f


def test_lazy_host_array_behaves_like_numpy():
    import torch
    from poor_man_gplvm_b200.hostio import LazyHostArray, to_numpy
    t = torch.arange(24, dtype=torch.float32).reshape(2, 3, 4) / 10
    a = LazyHostArray(t, torch.exp)
    want = np.exp(np.arange(24, dtype=np.float32).reshape(2, 3, 4) / 10)
    assert a.shape == (2, 3, 4) and a.ndim == 3 and len(a) == 2 and a.dtype == np.float32
    assert np.allclose(np.asarray(a), want)
    assert np.allclose(a[1, :, 2], want[1, :, 2])
    assert np.allclose(a - want, 0, atol=1e-5) and np.allclose(want - a, 0, atol=1e-5) and np.allclose(np.log(a), np.log(want))
    assert np.isclose(a.sum(), want.sum(), rtol=1e-5) and a.argmax() == want.argmax()
    assert np.array_equal(to_numpy(t), t.numpy())


# ----------------------------------------------------------------------------- jax.random bit streams (SURVEY F1)
def test_threefry_known_answers():
    """Random123 threefry2x32-20 known-answer vectors (also jax's own tests/random_test.py::testThreefry2x32)."""
    from poor_man_gplvm_b200 import jaxprng as jr
    def enc(k, c):
        a, b = jr.threefry2x32(k[0], k[1], np.uint32(c[0]), np.uint32(c[1]))
        return int(a), int(b)
    assert enc((0, 0), (0, 0)) == (0x6b200159, 0x99ba4efe)
    assert enc((0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff)) == (0x1cb996fc, 0xbb002be7)
    assert enc((0x13198a2e, 0x03707344), (0x243f6a88, 0x85a308d3)) == (0xc4923a9c, 0x483df7a0)


def test_jax_random_documented_values():
    """Values printed in the JAX documentation for PRNGKey(0) (recalled, JAX is not installable here):
    random.split(key) and the quickstart's random.normal(key, (10,))."""
    from poor_man_gplvm_b200 import jaxprng as jr
    key = jr.PRNGKey(0)
    assert jr.split(key).tolist() == [[4146024105, 967050713], [2718843009, 1272950319]]
    want = np.array([-0.3721109, 0.26423115, -0.18252768, -0.7368197, -0.44030377, -0.1521442, -0.67135346,
                     -0.5908641, 0.73168886, 0.5673026], dtype=np.float32)
    assert np.allclose(jr.normal(key, (10,)), want, rtol=0, atol=2e-7)
    u = jr.uniform(jr.PRNGKey(7), (5, 3))
    assert u.shape == (5, 3) and u.dtype == np.float32 and np.all((u >= 0) & (u < 1))
    # odd sizes use the padded counter layout
    assert np.array_equal(jr.random_bits(key, 5)[:2], jr.random_bits(key, 5)[:2])
    assert jr.random_bits(key, 5).shape == (5,)


def test_bench_reads_ncu_traffic_from_the_committed_profile():
    """bench.py reports `roofline.traffic` from the committed ncu --set full summary: the file must exist,
    parse, and carry the four hot kernels with plausible DRAM byte counts (headline workload)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    tr = bench.ncu_traffic()
    for k in ("emission_tc2_kernel", "atb_tc_kernel<1,0>", "atb_tc_kernel<2,1>", "fwd_c_kernel", "bwd_c_kernel"):
        assert k in tr, (k, sorted(tr))
        assert 1e9 < tr[k] < 2e10
    # emission moves its compulsory bytes (1 GB of fp16 counts in, 1.6 GB of ll out) and little more
    assert 2.4e9 < tr["emission_tc2_kernel"] < 3.0e9


def test_clock_sampler_parses_nvidia_smi_lines():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod2", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)

    class _P:
        def terminate(self): pass
        def kill(self): pass
        def communicate(self, timeout=None):
            return ("2026/10/18 12:00:00.100, 1965, 1965, 700.1, Not Active, Not Active, Not Active, Active\n"
                    "2026/10/18 12:00:00.200, 1800, 1965, 900.1, Not Active, Not Active, Not Active, Not Active\n"
                    "garbage line\n", "")
    s = bench.ClockSampler(0)
    s.proc = _P()
    out = s.stop()
    assert out["samples"] == 2 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]
    assert abs(out["sm_mhz"] - 1882.5) < 1e-6


def test_bench_dump_sample_and_format(tmp_path):
    """--dump-outputs: a fixed, sorted sample of distinct bins within the budget (all bins when they fit), float32
    kept, everything else stored as float64, and the 64 MB limit enforced before anything is written."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("bench_mod3", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rows = bench.dump_rows(10 ** 6, 4 * 400)
    assert len(rows) == bench.DUMP_TIME_BUDGET // 1600 and np.array_equal(rows, bench.dump_rows(10 ** 6, 1600))
    assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < 10 ** 6
    assert np.array_equal(bench.dump_rows(1000, 1600), np.arange(1000))
    bench.write_dump(str(tmp_path / "d"), {"a": torch.ones(3, 2), "n": 5, "h": torch.tensor(1.5, dtype=torch.float16),
                                           "bins": rows[:4]})
    got = {f[:-4]: np.load(tmp_path / "d" / f) for f in os.listdir(tmp_path / "d")}
    assert set(got) == {"a", "n", "h", "bins"} and got["a"].dtype == np.float32 and got["a"].shape == (3, 2)
    assert got["n"].dtype == got["h"].dtype == got["bins"].dtype == np.float64 and float(got["h"]) == 1.5
    with pytest.raises(RuntimeError):
        bench.write_dump(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()


def test_host_buffers_prefault_and_hand_out_arrays():
    """Result buffers are allocated up front and their pages populated on background threads (madvise pieces,
    memset fallback); take() returns the planned array once its pages are in, or None for an unplanned shape."""
    from poor_man_gplvm_b200 import hostio
    bufs = hostio.HostBuffers([("a", (1 << 20, 3), np.float32), ("b", (5, 7), np.float32)], threads=3)
    a = bufs.take("a")
    assert a.shape == (1 << 20, 3) and a.dtype == np.float32 and a.flags.c_contiguous
    a[:] = 1.5                                   # writable, fully mapped
    assert float(a.sum()) == 1.5 * a.size
    assert bufs.take("a") is None                # handed out once
    assert bufs.take("b", shape=(7, 5)) is None  # planned with another shape
    bufs.close()
    # a page-unaligned view in the middle of an array is handled (rounded down to the page, bounded by the view)
    x = np.zeros(3 * 4096 + 100, dtype=np.uint8)
    x[:] = 7
    hostio._touch(x[50:2 * 4096 + 77])
    assert int(x.min()) == 7 or int(x[50:2 * 4096 + 77].max()) in (0, 7)


def test_lazy_host_array_pickles_as_numpy():
    """em_res / decoding_res hold LazyHostArray objects (device tensors copied on first use); they must pickle to
    plain host data like the reference's jax arrays, including the ones built around a local producer."""
    import pickle
    import torch
    from poor_man_gplvm_b200 import hostio
    t = torch.arange(12, dtype=torch.float32).reshape(3, 4) + 1
    res = {"a": hostio.LazyHostArray(t, torch.log),
           "b": hostio.LazyHostArray(None, shape=(3, 4), producer=lambda: t * 2)}
    back = pickle.loads(pickle.dumps(res))
    assert isinstance(back["a"], np.ndarray) and isinstance(back["b"], np.ndarray)
    assert np.allclose(back["a"], np.log(t.numpy())) and np.array_equal(back["b"], (t * 2).numpy())


def test_circular_shuffle_and_latent_masks_on_host():
    """test.py:10-24 / model_selection_helper.py:249-254 helpers that need no GPU."""
    from poor_man_gplvm_b200 import test as shuf, model_selection_helper as msh
    y = np.arange(20, dtype=np.float32).reshape(5, 4)
    shifts = np.array([[0, 1, 2, 5], [3, 3, 3, 3]])
    out = list(shuf.circular_shuffle_data(y, n_shuffle=2, shifts=shifts))
    for i in range(2):
        for j in range(4):
            assert np.array_equal(out[i][:, j], np.roll(y[:, j], shifts[i, j]))
    masks = msh.draw_latent_masks(40, 0.2, 6, key=4)
    assert masks.shape == (6, 40) and set(np.unique(masks)) == {0.0, 1.0} and np.all(masks.sum(axis=1) == 8)
    assert np.array_equal(masks, msh.draw_latent_masks(40, 0.2, 6, key=4))
    e = shuf.compute_entropy(np.log(np.full((3, 2, 4), 1 / 8)))
    assert np.allclose(e, np.log(8))
    assert shuf.compute_entropy(np.array([[0.0, -np.inf]]), axis=-1)[0] == 0.0


def test_dense_scan_operand_pack_cpu():
    """Right-hand operands of the lockstep tensor-core scan (host-side packing, no GPU needed): the two fp16 pieces
    reconstruct 2^14 * P0 to 22 bits, the forward operand is the transpose of the backward one, padding is zero and
    the K-block ranges cover every non-zero of a block-banded kernel and skip the blocks outside the band."""
    from poor_man_gplvm_b200 import ops
    K = 300
    x = np.arange(K)
    dist = np.abs(x[:, None] - x[None, :])
    P0 = np.exp(-dist / 9.0) * (dist <= 40)
    P0 = P0 / P0.sum(axis=1, keepdims=True)
    d = ops.DenseMoveTC(P0, "cpu")
    assert (d.Kk, d.Kn, d.BN, d.n_ntiles) == (320, 320, 160, 2)
    buf = d.P16.numpy().astype(np.float64)
    rec = (buf[:, 0] + buf[:, 1]) / d.SCALE
    assert np.max(np.abs(rec[1, :K, :K] - P0)) <= 2.0 ** -22 * P0.max() * 1.01
    assert np.array_equal(buf[0, :, :K, :K], np.swapaxes(buf[1, :, :K, :K], 1, 2))
    assert not buf[:, :, K:].any() and not buf[:, :, :, K:].any()
    for dd in range(2):
        for i in range(d.n_ntiles):
            lo, hi = d.kb_host[dd, i]
            rows = rec[dd, i * d.BN:(i + 1) * d.BN]
            assert not rows[:, :lo * 64].any() and not rows[:, hi * 64:].any()
            assert rows[:, lo * 64:(lo + 1) * 64].any() and rows[:, (hi - 1) * 64:hi * 64].any()
    assert tuple(d.kb_host[0, 0]) == (0, 4) and tuple(d.kb_host[0, 1]) == (1, 5)
    assert ops.dense_scan_pays(2000, 1999) and not ops.dense_scan_pays(400, 5) and not ops.dense_scan_pays(100, 99)
