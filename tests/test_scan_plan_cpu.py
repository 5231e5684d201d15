"""CPU test: every scan entry point rejects a malformed chain plan, transition or mode with PMG_ERR_BAD_ARG.

The calls run in a subprocess that sees no CUDA device, so a call whose validation wrongly passes fails at its first
CUDA runtime call with a (positive) runtime error code instead of launching anything.  The lockstep (dense) passes get
no workspace: the workspace size is checked right after validation, so there a call that wrongly passes returns
PMG_ERR_WORKSPACE before it reaches any CUDA or driver call (their tensor-map setup would report a missing driver as
PMG_ERR_BAD_ARG).  The pointers are dummies: validation only tests them for NULL and alignment."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARG = -1
PMG_ERR_WORKSPACE = -4

SCRIPT = r"""
import ctypes as C, json
from poor_man_gplvm_b200 import _lib
from poor_man_gplvm_b200._lib import PmgScanPlan, PmgTransition
lib = _lib.load()
P = 1 << 20                       # dummy device pointer, 256-byte aligned
K = 64

def plan(**kw):
    p = PmgScanPlan()
    p.T, p.core_begin, p.core_end, p.chunk_len, p.n_chain, p.halo = 1000, 10, 1000, 100, 10, 20
    p.left_exact, p.right_exact, p.likelihood_scale, p.halo_next, p.sel_tol = 1, 1, 1.0, 0, 0.0
    p.sel_err = p.halo_arr = p.halo_next_arr = None
    for k, v in kw.items():
        setattr(p, k, v)
    return p

def trans(**kw):
    t = PmgTransition()
    t.K, t.kind, t.W, t.taps, t.inv_z, t.band_fwd, t.band_bwd = K, 0, 5, P, P, None, None
    for i, m in enumerate((0.99, 0.01, 0.01, 0.99)):
        t.M[i] = m
    for k, v in kw.items():
        setattr(t, k, v)
    return t

def call(name, pl, tr, a):
    r = lambda x: C.byref(x)
    ll, ldll, mode, ids, n_ids = a["ll"], a["ldll"], a["mode"], a["ids"], a["n_ids"]
    if name == "pmg_forward":
        return lib.pmg_forward(r(pl), r(tr), ll, ldll, None, None, 0, None, P, P, None, mode, ids, n_ids, None)
    if name == "pmg_backward":
        return lib.pmg_backward(r(pl), r(tr), ll, ldll, P, None, None, 0, None, P, None, None, 0, None, None, None,
                                None, None, mode, ids, n_ids, None)
    if name == "pmg_backward_xi16":
        return lib.pmg_backward_xi16(r(pl), r(tr), ll, ldll, P, None, None, 0, None, None, None, P, K, None, P, P, P,
                                     P, 2 * K, None, None, None, mode, ids, n_ids, None)
    if name == "pmg_forward_compact":
        return lib.pmg_forward_compact(r(pl), r(tr), ll, ldll, None, P, 0, None, P, K + 4, None, None, None, mode,
                                       ids, n_ids, None)
    if name == "pmg_backward_compact":
        return lib.pmg_backward_compact(r(pl), r(tr), ll, ldll, P, K + 4, None, P, 0, None, P, K, None, P, mode, ids,
                                        n_ids, None)
    if name == "pmg_forward_dense":
        return lib.pmg_forward_dense(r(pl), r(tr), P, None, 0, ll, ldll, None, None, 0, None, P, P, None, P, a["ws"],
                                     None)
    if name == "pmg_backward_dense":
        return lib.pmg_backward_dense(r(pl), r(tr), P, None, 0, ll, ldll, P, None, None, 0, None, None, None, None, 0,
                                      None, None, None, None, None, P, a["ws"], None)
    if name == "pmg_viterbi_forward":
        return lib.pmg_viterbi_forward(r(pl), r(tr), ll, ldll, None, P, 0, None, P, K, P, None, None, mode, ids,
                                       n_ids, None)
    if name == "pmg_viterbi_chain_maps":
        return lib.pmg_viterbi_chain_maps(r(pl), K, P, K, P, None)
    if name == "pmg_viterbi_backtrack":
        return lib.pmg_viterbi_backtrack(r(pl), K, P, K, P, P, P, None)
    if name == "pmg_viterbi_block_link":
        return lib.pmg_viterbi_block_link(r(pl), K, P, K, P, P, None)
    if name == "pmg_viterbi_backtrack_sharded":
        return lib.pmg_viterbi_backtrack_sharded(r(pl), K, P, K, P, P, 2, 0, P, None)
    raise KeyError(name)

FORWARD = {"pmg_forward", "pmg_forward_compact", "pmg_forward_dense", "pmg_viterbi_forward"}
out = {}
for name, entry in json.loads(ENTRIES).items():
    for case, (what, changes) in json.loads(CASES).items():
        if what not in entry:
            continue
        pk = dict(changes.get("plan", {}))
        tk = dict(changes.get("fwd_tr" if name in FORWARD else "bwd_tr", changes.get("tr", {})))
        a = dict(ll=P, ldll=K, mode=0, ids=None, n_ids=0, ws=0)
        a.update(changes.get("args", {}))
        out["%s/%s" % (name, case)] = call(name, plan(**pk), trans(**tk), a)
print(json.dumps(out))
"""

# entry point -> what it takes besides the plan: a transition (with ll and ldll) and a repair mode
ENTRIES = {
    "pmg_forward": ["plan", "tr", "mode"],
    "pmg_backward": ["plan", "tr", "mode"],
    "pmg_backward_xi16": ["plan", "tr", "mode"],
    "pmg_forward_compact": ["plan", "tr", "mode"],
    "pmg_backward_compact": ["plan", "tr", "mode"],
    "pmg_forward_dense": ["plan", "tr"],
    "pmg_backward_dense": ["plan", "tr"],
    "pmg_viterbi_forward": ["plan", "tr", "mode"],
    "pmg_viterbi_chain_maps": ["plan"],
    "pmg_viterbi_backtrack": ["plan"],
    "pmg_viterbi_block_link": ["plan"],
    "pmg_viterbi_backtrack_sharded": ["plan"],
}
# case -> (argument it breaks, changes to the well-formed call); the base plan has 10 chains of 100 bins over the
# 990 core bins [10, 1000) of T = 1000
CASES = {
    "core_end_past_T": ("plan", {"plan": {"core_end": 1001}}),
    "chunk_len_zero": ("plan", {"plan": {"chunk_len": 0}}),
    "too_few_chains": ("plan", {"plan": {"n_chain": 9}}),
    "empty_trailing_chain": ("plan", {"plan": {"n_chain": 11}}),
    "negative_halo": ("plan", {"plan": {"halo": -1}}),
    "negative_halo_next": ("plan", {"plan": {"halo_next": -1}}),
    "mode_3": ("mode", {"args": {"mode": 3}}),
    "mode_1_without_ids": ("mode", {"args": {"mode": 1}}),
    "mode_2_without_sel_err": ("mode", {"args": {"mode": 2}}),
    "kind_2": ("tr", {"tr": {"kind": 2}}),
    "kind_0_without_taps": ("tr", {"tr": {"taps": None}}),
    "kind_1_without_the_band_of_its_direction": ("tr", {"fwd_tr": {"kind": 1, "band_bwd": 1 << 20},
                                                        "bwd_tr": {"kind": 1, "band_fwd": 1 << 20}}),
    "W_above_K_minus_1": ("tr", {"tr": {"W": 64}}),
    "ldll_below_K": ("tr", {"args": {"ldll": 63}}),
}


def _run(entries, cases):
    from poor_man_gplvm_b200 import build
    build.build()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=ROOT)
    code = "ENTRIES = %r\nCASES = %r\n" % (json.dumps(entries), json.dumps(cases)) + SCRIPT
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.fixture(scope="module")
def results():
    return _run(ENTRIES, dict(CASES, well_formed=("plan", {})))


def test_every_scan_entry_point_rejects_malformed_plans(results):
    wrong = {k: v for k, v in results.items() if not k.endswith("/well_formed") and v != BAD_ARG}
    assert not wrong, wrong
    for name, entry in ENTRIES.items():
        n = sum(what in entry for what, _ in CASES.values())
        assert sum(k.startswith(name + "/") for k in results) == n + 1, name


def test_a_well_formed_plan_passes_validation(results):
    # past validation, the first CUDA runtime call finds no device: a positive cudaError_t
    got = {k: v for k, v in results.items() if k.endswith("/well_formed")}
    assert len(got) == len(ENTRIES)
    for k, v in got.items():
        if "_dense/" in k:
            assert v == PMG_ERR_WORKSPACE, got
        else:
            assert v > 0, got
