"""ctypes binding of libpmgplvm_b200.so (the C ABI declared in include/pmgplvm_b200.h).

There is no CPU or PyTorch fallback: if the library cannot be loaded every
operator raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpmgplvm_b200.so")

c_f32p = C.c_void_p   # device pointers travel as integers
c_i32p = C.c_void_p
c_i32p_host = C.POINTER(C.c_int)   # host int arrays / out-parameters
c_stream = C.c_void_p


class PmgTransition(C.Structure):
    _fields_ = [("K", C.c_int), ("kind", C.c_int), ("W", C.c_int),
                ("taps", C.c_void_p), ("inv_z", C.c_void_p),
                ("band_fwd", C.c_void_p), ("band_bwd", C.c_void_p),
                ("M", C.c_float * 4)]


class PmgScanPlan(C.Structure):
    _fields_ = [("T", C.c_int64), ("core_begin", C.c_int64), ("core_end", C.c_int64),
                ("chunk_len", C.c_int64), ("n_chain", C.c_int), ("halo", C.c_int),
                ("left_exact", C.c_int), ("right_exact", C.c_int),
                ("likelihood_scale", C.c_float), ("halo_next", C.c_int), ("sel_tol", C.c_float),
                ("sel_err", C.c_void_p), ("halo_arr", C.c_void_p), ("halo_next_arr", C.c_void_p)]


# name -> (restype, argtypes); must list every symbol declared in include/pmgplvm_b200.h
SIGNATURES = {
    "pmg_version": (C.c_int, []),
    "pmg_error_string": (C.c_char_p, [C.c_int]),
    "pmg_sm_count": (C.c_int, []),
    "pmg_emission_prepare": (C.c_int, [C.c_int, C.c_int, c_f32p, c_f32p, C.c_float, c_f32p, c_f32p, c_stream]),
    "pmg_emission_lgamma_rowsum": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, c_stream]),
    "pmg_emission_row_terms": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p, c_f32p,
                                         c_stream]),
    "pmg_emission_prepare_aug": (C.c_int, [C.c_int, C.c_int, c_f32p, c_f32p, C.c_float, C.c_int, C.c_int, c_f32p,
                                           C.c_int64, c_f32p, c_stream]),
    "pmg_emission_poisson": (C.c_int, [C.c_int64, C.c_int, C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p,
                                       c_f32p, c_f32p, C.c_int64, c_stream]),
    "pmg_emission_gaussian": (C.c_int, [C.c_int64, C.c_int, C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64,
                                        C.c_float, c_f32p, c_f32p, C.c_int64, c_stream]),
    "pmg_counts_prepare": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_void_p, C.c_int64, C.c_int,
                                     c_i32p, c_f32p, c_f32p, c_stream]),
    "pmg_counts_prepare_shifted": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, c_i32p, c_f32p,
                                             C.c_void_p, C.c_int64, c_f32p, c_stream]),
    "pmg_counts_to_f16": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, C.c_void_p, C.c_int64, c_i32p, c_stream]),
    "pmg_emission_tile_n": (C.c_int, [C.c_int]),
    "pmg_emission_prepare_f16": (C.c_int, [C.c_int, C.c_int, c_f32p, c_f32p, C.c_float, C.c_int, C.c_int64,
                                           C.c_void_p, c_f32p, c_stream]),
    "pmg_emission_poisson_f16": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int,
                                           c_f32p, c_f32p, c_f32p, c_f32p, C.c_int64, c_stream]),
    "pmg_naive_bayes_normalize": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p,
                                            c_stream]),
    "pmg_naive_bayes_lml": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, c_stream]),
    "pmg_naive_bayes_posterior": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p,
                                            c_stream]),
    "pmg_forward": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                              c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, c_i32p, C.c_int, c_stream]),
    "pmg_backward": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                               c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                               C.c_int, c_i32p, C.c_int, c_stream]),
    "pmg_viterbi_forward": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                                      c_f32p, C.c_int64, c_f32p, C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p,
                                      C.c_int, c_i32p, C.c_int, c_stream]),
    "pmg_viterbi_chain_maps": (C.c_int, [C.POINTER(PmgScanPlan), C.c_int, C.c_void_p, C.c_int64, c_i32p,
                                         c_stream]),
    "pmg_viterbi_backtrack": (C.c_int, [C.POINTER(PmgScanPlan), C.c_int, C.c_void_p, C.c_int64, c_i32p, c_f32p,
                                        c_i32p, c_stream]),
    "pmg_viterbi_block_link": (C.c_int, [C.POINTER(PmgScanPlan), C.c_int, C.c_void_p, C.c_int64, c_i32p, c_i32p,
                                         c_stream]),
    "pmg_viterbi_backtrack_sharded": (C.c_int, [C.POINTER(PmgScanPlan), C.c_int, C.c_void_p, C.c_int64, c_i32p,
                                                c_i32p, C.c_int, C.c_int, c_i32p, c_stream]),
    "pmg_dense_scan_geometry":(C.c_int, [C.c_int, c_i32p_host, c_i32p_host, c_i32p_host, c_i32p_host]),
    "pmg_dense_scan_workspace_bytes": (C.c_int64, [C.c_int, C.c_int]),
    "pmg_forward_dense": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), C.c_void_p, c_i32p_host,
                                    C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p,
                                    c_f32p, C.c_void_p, C.c_int64, c_stream]),
    "pmg_backward_dense": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), C.c_void_p, c_i32p_host,
                                     C.c_int, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p,
                                     c_f32p, C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                     C.c_void_p, C.c_int64, c_stream]),
    "pmg_backward_xi16_supported": (C.c_int, [C.POINTER(PmgTransition), C.c_float]),
    "pmg_backward_xi16": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                                    c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_void_p, C.c_int64, c_f32p,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, c_f32p, c_f32p, c_f32p,
                                    C.c_int, c_i32p, C.c_int, c_stream]),
    "pmg_atb_bf16x2_pieces": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                        C.c_void_p, C.c_int64, c_f32p, C.c_void_p, C.c_int64, c_stream]),
    "pmg_boundary_pack_fwd": (C.c_int, [C.c_int, c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, c_f32p, C.c_float, c_f32p,
                                        c_stream]),
    "pmg_boundary_unpack_fwd": (C.c_int, [C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, c_f32p, c_f32p, C.c_float,
                                          c_f32p, c_stream]),
    "pmg_scan_compact_supported": (C.c_int, [C.POINTER(PmgTransition), C.c_float]),
    "pmg_forward_compact": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                                      c_f32p, C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, c_f32p, c_f32p, C.c_int,
                                      c_i32p, C.c_int, c_stream]),
    "pmg_backward_compact": (C.c_int, [C.POINTER(PmgScanPlan), C.POINTER(PmgTransition), c_f32p, C.c_int64, c_f32p,
                                       C.c_int64, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_void_p, C.c_int64,
                                       c_f32p, c_f32p, C.c_int, c_i32p, C.c_int, c_stream]),
    "pmg_split_f16": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, C.c_void_p, C.c_int64, c_stream]),
    "pmg_split_bf16": (C.c_int, [C.c_int64, C.c_int, c_f32p, C.c_int64, C.c_void_p, C.c_int64, c_stream]),
    "pmg_atb_bf16x2": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, c_f32p,
                                 C.c_void_p, C.c_int64, c_stream]),
    "pmg_atb_f16_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int, C.c_int]),
    "pmg_atb_f16": (C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, c_f32p,
                              C.c_void_p, C.c_int64, c_stream]),
    "pmg_seam_check": (C.c_int, [C.c_int, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_int64, C.c_float, c_f32p,
                                 c_stream]),
    "pmg_seam_check_fix": (C.c_int, [C.c_int, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_int64, C.c_float, C.c_float,
                                     C.c_int, c_f32p, c_f32p, c_stream]),
    "pmg_strided_sum_workspace_bytes": (C.c_int64, []),
    "pmg_strided_sum": (C.c_int, [C.c_int64, c_f32p, C.c_int64, c_f32p, C.c_void_p, c_stream]),
    "pmg_atb_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int, C.c_int, C.c_int]),
    "pmg_atb": (C.c_int, [C.c_int64, C.c_int, C.c_int, c_f32p, C.c_int64, c_f32p, C.c_int64, c_f32p, C.c_int64,
                          C.c_void_p, C.c_int64, C.c_int, c_stream]),
    "pmg_xi_finalize": (C.c_int, [C.c_int, c_f32p, c_f32p, C.POINTER(C.c_float), c_f32p, c_stream]),
    "pmg_mstep_workspace_bytes": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "pmg_mstep_adam": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, C.c_float, C.c_float,
                                 C.c_float, C.c_float, C.c_float, C.c_int, C.c_float, C.c_int, c_f32p, c_f32p,
                                 c_f32p, c_i32p, c_f32p, c_f32p, c_i32p, c_f32p, c_f32p, C.c_void_p, C.c_int64,
                                 c_stream]),
    "pmg_mstep_adam_ld": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, C.c_int64, c_f32p, C.c_int64,
                                    C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int, C.c_float,
                                    C.c_int, c_f32p, c_f32p, c_f32p, c_i32p, c_f32p, c_f32p, c_i32p, c_f32p, c_f32p,
                                    C.c_void_p, C.c_int64, c_stream]),
    "pmg_mstep_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_i32p_host, c_i32p_host, c_i32p_host,
                                 c_i32p_host]),
    "pmg_threefry_posterior_init": (C.c_int, [C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_uint32, C.c_uint32,
                                              C.c_float, c_f32p, C.c_int64, c_f32p, C.c_int64, C.c_void_p, C.c_int64,
                                              C.c_int64, C.c_void_p, c_stream]),
    "pmg_tuning_softplus": (C.c_int, [C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_stream]),
}

_lib = None


def load():
    """Load the shared library (once) and attach prototypes.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "poor_man_gplvm_b200: %s not found. Build it with `python -m poor_man_gplvm_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class PmgError(RuntimeError):
    pass


def check(code, what):
    if code != 0:
        msg = load().pmg_error_string(int(code)).decode()
        raise PmgError("%s failed: %s (code %d)" % (what, msg, code))
