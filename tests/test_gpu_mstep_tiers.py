"""The Adam M-step (csrc/pmg_mstep.cu) at every kernel and dispatch tier, against the fp64 optimiser
oracle.ref_numpy.adam_run.

The launch picks one of two cooperative kernels and a placement of Phi from the shapes and the device's occupancy
(ops.mstep_plan reports the choice; each case asserts the tier it was written for and skips, naming the plan, when
the device places it elsewhere):

  lag-smem       lagged kernel, Phi in shared memory, gradient K sum split into parts = 512/B > 1
  lag-global     lagged kernel, Phi in global memory (K*B too large for shared memory), parts >= 2
  lag-parts1     lagged kernel, 256 < B < 512: one gradient part, threads tid < B
  barrier-smem   barrier kernel, Phi in shared memory, one tile per CTA
  barrier-wide   barrier kernel, Phi in global memory, B >= 256 (the lagged kernel's ring does not fit)
  barrier-multi  barrier kernel, more tiles of 4 neurons than resident CTAs: each CTA loops over several

Every case makes two consecutive calls (the second continues the optimiser state, count > 0) and checks, per call:
n_iter and count exactly; loss / error history zero past n_iter; final = the last history entry, bit for bit;
W, mu, nu, loss history, error history and final against fp64; tuning_out against softplus(Phi W) evaluated in
fp64 from the kernel's own W, and ops.tuning_softplus bit for bit; canary words around every output buffer.

Tolerances.  Adam's m/sqrt(v) amplifies rounding, so W, mu, nu and the histories are held to the fp32 reference's own
distance from fp64 (adam_run on float32 inputs, same calls):  max|gpu - fp64| <= SPREAD * max|fp32 - fp64| +
FLOOR * max|fp64|, with SPREAD = 8 and FLOOR = 2e-5 (1e-5 for the loss).  A ring slot one step off moves W by about
lr = 0.01 and mu by ~10 %, orders of magnitude above either bound.  On the CPU, the fp32 reference's own spread is
1e-6 to 7e-5 of max|x| over these cases, so the floor dominates the bound in most of them.
tuning_out is held to a rounding bound that does not depend on the optimiser: |tuning - softplus(z)| <=
sigmoid(z) * B * 2^-24 * sum_b |Phi W| + 8 * 2^-24 * softplus(z), z = Phi W in fp64.
The module prints the largest error / bound of each quantity over all cases when it ends.
"""
import contextlib
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

torch = pytest.importorskip("torch")

from oracle import ref_numpy as ref

pytestmark = pytest.mark.gpu

PRIOR_STD, LR = 1.0, 0.01
SPREAD, FLOOR, FLOOR_LOSS = 8.0, 2e-5, 1e-5
U32 = 2.0 ** -24
CANARY = -1.2345e30
PAD = 64          # canary words before and after every output buffer
MARGINS = {}      # quantity -> largest error / bound seen, reported at the end of the module


@pytest.fixture(scope="module")
def ops(request):
    from poor_man_gplvm_b200 import ops as _ops
    yield _ops
    _log(request, "mstep tiers: largest error/bound " +
         ", ".join("%s %.3g" % kv for kv in sorted(MARGINS.items())))


@pytest.fixture(scope="module")
def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _log(request, msg):
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    if tr is not None:
        tr.write_line(msg)
    else:
        print(msg)


@contextlib.contextmanager
def lag_env(lag):
    """PMG_MSTEP_LAG for the launches inside (None: the production default)."""
    old = os.environ.get("PMG_MSTEP_LAG")
    if lag is not None:
        os.environ["PMG_MSTEP_LAG"] = lag
    try:
        yield
    finally:
        os.environ.pop("PMG_MSTEP_LAG", None)
        if old is not None:
            os.environ["PMG_MSTEP_LAG"] = old


def estep_stats(K, N, ls, seed):
    """Basis and E-step-like statistics: tw_k in [1, 50] (posterior mass of latent bin k), yw_kn ~ tw_k * lambda_kn
    with bump-shaped rates and some exact zeros (a neuron silent at that latent position)."""
    rng = np.random.default_rng(seed)
    basis = ref.generate_basis(ls, K, dtype=np.float32)
    B = basis.shape[1]
    tw = (1.0 + 49.0 * rng.random(K)).astype(np.float32)
    x = np.arange(K)[:, None] / max(K - 1, 1)
    lam = 0.02 + 3.0 * rng.random(N) * np.exp(-0.5 * ((x - rng.random(N)) / (0.05 + 0.3 * rng.random(N))) ** 2)
    yw = tw[:, None] * lam * rng.gamma(4.0, 0.25, size=(K, N))
    yw[rng.random((K, N)) < 0.15] = 0.0
    W0 = (0.3 * rng.standard_normal((B, N))).astype(np.float32)
    return basis, yw.astype(np.float32), tw, W0


def _padded(shape, dtype=torch.float32):
    n = int(np.prod(shape))
    buf = torch.full((PAD + n + PAD,), CANARY, dtype=dtype, device="cuda")
    return buf, buf[PAD:PAD + n].view(shape)


def _canaries_intact(buf):
    h = buf.cpu().numpy()
    return bool(np.all(h[:PAD] == CANARY) and np.all(h[-PAD:] == CANARY))


class GpuRun:
    """W, mu, nu, count on the device in canaried buffers; calls ops.mstep_adam with canaried outputs."""

    def __init__(self, ops, W0):
        B, N = W0.shape
        self.ops = ops
        self.bufs = {}
        for nm in ("W", "mu", "nu"):
            self.bufs[nm], t = _padded((B, N))
            t.copy_(torch.from_numpy(W0) if nm == "W" else torch.zeros(B, N))
            setattr(self, nm, t)
        self.state = ops.AdamState(self.W)
        self.state.mu, self.state.nu = self.mu, self.nu

    def call(self, Phi, yw, tw, maxiter, tol, min_iters):
        K, N = Phi.shape[0], self.W.shape[1]
        outs = {nm: _padded(shape) for nm, shape in (("lh", (maxiter,)), ("eh", (maxiter,)), ("fin", (2,)),
                                                     ("tuning", (K, N)))}
        n_iter = torch.full((1,), -7, dtype=torch.int32, device="cuda")
        self.ops.mstep_adam(Phi, yw, tw, self.W, self.state, PRIOR_STD, LR, maxiter, tol, min_iters=min_iters,
                            out=(outs["lh"][1], outs["eh"][1], n_iter, outs["fin"][1], outs["tuning"][1]))
        torch.cuda.synchronize()
        got = {nm: o[1].cpu().numpy().copy() for nm, o in outs.items()}
        got.update(n_iter=int(n_iter.item()), count=int(self.state.count.item()),
                   W=self.W.cpu().numpy().copy(), mu=self.mu.cpu().numpy().copy(), nu=self.nu.cpu().numpy().copy())
        bad = [nm for nm, o in outs.items() if not _canaries_intact(o[0])]
        bad += [nm for nm, b in self.bufs.items() if not _canaries_intact(b)]
        assert not bad, "writes outside the output buffers: %s" % bad
        got["tuning_op"] = self.ops.tuning_softplus(Phi, self.W).cpu().numpy()
        return got


def _bound_check(name, got, want64, want32, floor):
    err = float(np.max(np.abs(got.astype(np.float64) - want64)))
    spread = float(np.max(np.abs(want32.astype(np.float64) - want64)))
    bound = SPREAD * spread + floor * max(float(np.max(np.abs(want64))), 1e-30)
    MARGINS[name] = max(MARGINS.get(name, 0.0), err / bound)
    assert err <= bound, "%s: max|gpu - fp64| = %.3g > %g * %.3g (fp32 spread) + floor = %.3g" % (
        name, err, SPREAD, spread, bound)


def check_call(got, w64, w32, basis, maxiter, n_expect):
    """One M-step call against the fp64 run w64 and the fp32 run w32 of adam_run from the same state."""
    n = got["n_iter"]
    assert n == n_expect == w64["n_iter"], (n, n_expect, w64["n_iter"])
    assert got["count"] == w64["opt_state"]["count"]
    assert np.all(got["lh"][n:] == 0) and np.all(got["eh"][n:] == 0), "history written past n_iter"
    assert got["fin"][0] == got["lh"][n - 1] and got["fin"][1] == got["eh"][n - 1]
    _bound_check("loss", got["lh"][:n], w64["loss_history"][:n], w32["loss_history"][:n], FLOOR_LOSS)
    _bound_check("err", got["eh"][:n], w64["error_history"][:n], w32["error_history"][:n], FLOOR)
    _bound_check("W", got["W"], w64["params"], w32["params"], FLOOR)
    _bound_check("mu", got["mu"], w64["opt_state"]["mu"], w32["opt_state"]["mu"], FLOOR)
    _bound_check("nu", got["nu"], w64["opt_state"]["nu"], w32["opt_state"]["nu"], FLOOR)
    # tuning_out = softplus(Phi W) of the kernel's own final W: a rounding bound independent of the optimiser
    Phi64, Wg = basis.astype(np.float64), got["W"].astype(np.float64)
    z = Phi64 @ Wg
    sp = ref.softplus(z)
    bound = (1.0 / (1.0 + np.exp(-z))) * basis.shape[1] * U32 * (np.abs(Phi64) @ np.abs(Wg)) + 8 * U32 * sp + 1e-37
    ratio = np.abs(got["tuning"] - sp) / bound
    MARGINS["tuning"] = max(MARGINS.get("tuning", 0.0), float(ratio.max()))
    assert np.all(ratio <= 1.0), "tuning_out off softplus(Phi W) by %.3g x the rounding bound" % ratio.max()
    assert np.array_equal(got["tuning_op"], got["tuning"]), "ops.tuning_softplus differs from the M-step's tuning"


def oracle_pair(basis, yw, tw, state64, state32, maxiter, tol, min_iters):
    """adam_run in fp64 and in fp32, each continuing its own previous state (W, opt_state)."""
    out = []
    for (W, opt), dt in ((state64, np.float64), (state32, np.float32)):
        out.append(ref.adam_run(W, opt, PRIOR_STD, basis.astype(dt), yw.astype(dt), tw.astype(dt), step_size=LR,
                                maxiter=maxiter, tol=tol, min_iters=min_iters))
    return out


def run_two_calls(ops, basis, yw, tw, W0, calls):
    """calls: [(maxiter, tol, min_iters, n_expect)] made one after the other from W0 and a fresh optimiser."""
    Phi, ywd, twd = (torch.from_numpy(a).cuda() for a in (basis, yw, tw))
    run = GpuRun(ops, W0)
    s64 = (W0.astype(np.float64), ref.adam_init(W0.astype(np.float64)))
    s32 = (W0.copy(), ref.adam_init(W0.copy()))
    results = []
    for maxiter, tol, min_iters, n_expect in calls:
        before = {nm: getattr(run, nm).cpu().numpy().copy() for nm in ("W", "mu", "nu")}
        count_before = int(run.state.count.item())
        got = run.call(Phi, ywd, twd, maxiter, tol, min_iters)
        w64, w32 = oracle_pair(basis, yw, tw, s64, s32, maxiter, tol, min_iters)
        check_call(got, w64, w32, basis, maxiter, n_expect)
        results.append((got, before, count_before))
        s64 = (w64["params"], w64["opt_state"])
        s32 = (w32["params"], w32["opt_state"])
    return results


# ----------------------------------------------------------------------------- tier matrix
def _tier_ok(tier, plan, B):
    if tier == "lag-smem":
        return plan["kernel"] == "lagged" and plan["phi_in_smem"] and plan["parts"] > 1
    if tier == "lag-global":
        return plan["kernel"] == "lagged" and not plan["phi_in_smem"] and plan["parts"] >= 2
    if tier == "lag-parts1":
        return plan["kernel"] == "lagged" and plan["parts"] == 1 and 256 < B < 512
    if tier == "barrier-smem":
        return plan["kernel"] == "barrier" and plan["phi_in_smem"] and plan["tiles_per_cta"] == 1
    if tier == "barrier-wide":
        return (plan["kernel"] == "barrier" and not plan["phi_in_smem"] and B >= 256 and plan["parts"] == 1
                and plan["tiles_per_cta"] == 1)
    if tier == "barrier-multi":
        return plan["kernel"] == "barrier" and plan["tiles_per_cta"] >= 2
    raise AssertionError(tier)


# (tier, K, lengthscale, N, PMG_MSTEP_LAG); N "4sm" / "4sm+1" = 4 neurons per SM of this device (+1)
TIER_CASES = [
    ("lag-smem", 400, 10.0, 500, None),          # headline shape
    ("lag-smem", 100, 10.0, 33, None),
    ("lag-smem", 200, 10.0, "4sm", None),        # every SM holds one CTA of the lagged kernel
    ("lag-smem", 3, 5.0, 1, None),               # tiny
    ("lag-global", 1000, 10.0, 250, None),       # B = 151
    ("lag-parts1", 512, 2.0, 150, None),         # B = 381
    ("barrier-smem", 200, 10.0, "4sm+1", None),  # one tile more than the lagged kernel can hold
    ("barrier-smem", 400, 10.0, 500, "0"),
    ("barrier-smem", 100, 10.0, 33, "0"),
    ("barrier-wide", 2000, 10.0, 300, None),     # config E, B = 299
    ("barrier-wide", 600, 1.0, 37, None),        # B = 600
    ("barrier-wide", 2000, 3.0, 21, None),       # B = 990
    ("barrier-multi", 400, 10.0, 3001, None),
    ("barrier-multi", 50, 5.0, 4999, None),      # B = 17, several tiles per CTA
]


@pytest.mark.parametrize("tier,K,ls,N,lag", TIER_CASES,
                         ids=["%s-K%d-N%s%s" % (t, K, N, "-lag0" if lag else "") for t, K, ls, N, lag in TIER_CASES])
def test_mstep_tier_matches_fp64(ops, n_sm, request, tier, K, ls, N, lag):
    N = {"4sm": 4 * n_sm, "4sm+1": 4 * n_sm + 1}.get(N, N)
    basis, yw, tw, W0 = estep_stats(K, N, ls, seed=K * 7919 + N)
    B = basis.shape[1]
    with lag_env(lag):
        plan = ops.mstep_plan(K, B, N, 24)
        _log(request, "mstep plan %s K=%d B=%d N=%d (%d SMs): %s" % (tier, K, B, N, n_sm, plan))
        if not _tier_ok(tier, plan, B):
            pytest.skip("this device places K=%d B=%d N=%d on %s, not on tier %s" % (K, B, N, plan, tier))
        # tol = -1: every call runs exactly maxiter - 1 updates; 24 and 11 steps wrap the 9-slot ring
        run_two_calls(ops, basis, yw, tw, W0, [(24, -1.0, 5, 24), (11, -1.0, 5, 11)])


# ----------------------------------------------------------------------------- stop-rule edges
# deterministic rules (the stop step is decided by the rule, never by rounding):
#   tol -1           never stops early: n_iter = maxiter
#   tol 1e30         stops at min_iters = 5 (the lagged kernel has run up to 7 steps ahead: ring restore)
#   tol 0, min 1     the second loss is the first one again (the loss lags W by one update): n_iter = 2
#   tol 1e30, min 0  stops before the first update: W, mu, nu and count untouched
RULES = {"tol-1": (-1.0, 5), "tol1e30": (1e30, 5), "tol0-min1": (0.0, 1), "min0": (1e30, 0)}


def _n_expect(rule, maxiter):
    return {"tol-1": maxiter, "tol1e30": min(maxiter, 6), "tol0-min1": min(maxiter, 2), "min0": 1}[rule]


@pytest.mark.parametrize("kernel", ["lagged", "barrier"])
@pytest.mark.parametrize("rule", list(RULES))
@pytest.mark.parametrize("maxiter", [1, 2, 3, 5, 6, 9, 10, 14])
def test_mstep_stop_rule_edges(ops, request, kernel, rule, maxiter):
    K, N, ls = 64, 30, 4.0
    basis, yw, tw, W0 = estep_stats(K, N, ls, seed=11)
    B = basis.shape[1]
    tol, min_iters = RULES[rule]
    n = _n_expect(rule, maxiter)
    with lag_env("0" if kernel == "barrier" else None):
        plan = ops.mstep_plan(K, B, N, maxiter)
        if plan["kernel"] != kernel:
            pytest.skip("this device places K=%d B=%d N=%d on %s" % (K, B, N, plan))
        res = run_two_calls(ops, basis, yw, tw, W0, [(maxiter, tol, min_iters, n), (maxiter, tol, min_iters, n)])
    for got, before, count_before in res:
        assert got["count"] == count_before + n - 1
        if rule == "tol0-min1" and maxiter >= 2:
            assert got["lh"][1] == got["lh"][0]
        if rule == "min0":
            for nm in ("W", "mu", "nu"):
                assert np.array_equal(got[nm], before[nm]), nm


# ----------------------------------------------------------------------------- production layout
@pytest.mark.parametrize("kernel", ["lagged", "barrier"])
def test_mstep_statistics_view_bit_identical(ops, kernel):
    """yw / tw as the [K, N+1] statistics buffer EMLoop passes (yw = stats[:, :N], tw = stats[:, N], both with row
    stride N+1) give the same bits as contiguous copies."""
    K, N, ls = 400, 501, 10.0
    basis, yw, tw, W0 = estep_stats(K, N, ls, seed=5)
    B = basis.shape[1]
    with lag_env("0" if kernel == "barrier" else None):
        plan = ops.mstep_plan(K, B, N, 40)
        if plan["kernel"] != kernel:
            pytest.skip("this device places K=%d B=%d N=%d on %s" % (K, B, N, plan))
        Phi = torch.from_numpy(basis).cuda()
        stats = torch.from_numpy(np.concatenate([yw, tw[:, None]], axis=1)).cuda()
        outs = []
        for ywd, twd in ((stats[:, :N], stats[:, N]), (stats[:, :N].contiguous(), stats[:, N].contiguous())):
            run = GpuRun(ops, W0)
            res = [run.call(Phi, ywd, twd, 40, 1e-6, 5) for _ in range(2)]
            outs.append(res)
    assert outs[0][0]["n_iter"] >= 6
    for a, b in zip(*outs):
        for nm in ("lh", "eh", "fin", "tuning", "W", "mu", "nu", "n_iter", "count"):
            assert np.array_equal(a[nm], b[nm]), nm


# ----------------------------------------------------------------------------- argument errors
def test_mstep_argument_errors_launch_nothing(ops):
    from poor_man_gplvm_b200 import _lib
    lib = _lib.load()
    K, N, ls = 64, 30, 4.0
    basis, yw, tw, W0 = estep_stats(K, N, ls, seed=3)
    B = basis.shape[1]
    Phi, ywd, twd = (torch.from_numpy(a).cuda() for a in (basis, yw, tw))
    run = GpuRun(ops, W0)
    maxiter = 10
    lh, eh, fin = (torch.full((n,), 7.0, device="cuda") for n in (maxiter, maxiter, 2))
    tun = torch.full((K, N), 7.0, device="cuda")
    n_iter = torch.full((1,), -7, dtype=torch.int32, device="cuda")
    need = lib.pmg_mstep_workspace_bytes(K, B, N, maxiter)
    ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(mi, nbytes):
        return lib.pmg_mstep_adam_ld(K, B, N, p(Phi), p(ywd), N, p(twd), 1, PRIOR_STD, LR, 0.9, 0.999, 1e-8, mi, -1.0,
                                     5, p(run.W), p(run.mu), p(run.nu), p(run.state.count), p(lh), p(eh), p(n_iter),
                                     p(fin), p(tun), p(ws), nbytes, stream)

    assert call(0, need) == -1                        # PMG_ERR_BAD_ARG
    assert call(maxiter, need - 1) == -4              # PMG_ERR_WORKSPACE
    assert lib.pmg_mstep_plan(K, B, N, 0, None, None, None, None) == -1
    torch.cuda.synchronize()
    for t in (lh, eh, fin, tun):
        assert bool(torch.all(t == 7.0))
    assert int(n_iter.item()) == -7 and int(run.state.count.item()) == 0
    assert np.array_equal(run.W.cpu().numpy(), W0) and not bool(run.mu.any()) and not bool(run.nu.any())
    assert int(ws.sum().item()) == 0
    # the same buffers with a valid call do run
    assert call(maxiter, need) == 0
    torch.cuda.synchronize()
    assert int(n_iter.item()) == maxiter
