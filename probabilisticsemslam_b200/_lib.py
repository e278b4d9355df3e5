"""Loads libpda_b200.so (the CUDA product) and declares its C ABI (include/pda_b200.h).

There is no fallback of any kind: if the shared library is missing or a call fails the
caller gets an exception.  The oracle under oracle/ is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PDA_B200_LIB", os.path.join(_HERE, "libpda_b200.so"))  # override: A/B builds while tuning

i32, i64, u64, dbl, ptr = C.c_int32, C.c_int64, C.c_uint64, C.c_double, C.c_void_p

# name -> (restype, argtypes); kept in the order of include/pda_b200.h
SIGNATURES = {
    "pda_version": (C.c_int, []),
    "pda_last_error": (C.c_char_p, []),
    "pda_device_count": (C.c_int, []),
    "pda_diag_dfma_tflops": (dbl, []),
    "pda_host_alloc": (ptr, [i64]),
    "pda_host_free": (None, [ptr]),
    "pda_murty_workspace_bytes": (i64, [i64, i32, i32, i32]),
    "pda_murty_set_path": (C.c_int, [i32]),
    "pda_murty_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, i32, i32, i32, dbl, i32, i32,
                                  ptr, ptr, ptr, ptr, ptr, ptr, i32, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_murty_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, i32, dbl, i32, i32,
                                       ptr, ptr, ptr, ptr, ptr, ptr, i32, ptr, ptr, ptr, i32]),
    "pda_murty_batch_host_multi": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, i32, dbl, i32, i32,
                                             ptr, ptr, ptr, ptr, ptr, ptr, i32, ptr, ptr, ptr, ptr, i32]),
    "pda_assignment_prob_ladder_batch": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, i32, i32, ptr, i32, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_assignment_prob_ladder_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, ptr, i32, ptr, ptr, ptr, i32]),
    "pda_lap_batch": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, i32, i32, i32, i32, ptr, ptr,
                                ptr, ptr, ptr, ptr, ptr, ptr, ptr, ptr]),
    "pda_lap_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, i32, i32, ptr, ptr,
                                     ptr, ptr, ptr, ptr, ptr, ptr, ptr, i32]),
    "pda_condition_costs_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, ptr]),
    "pda_condition_costs_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, i32]),
    "pda_to_probs_batch": (C.c_int, [ptr, ptr, ptr, i64, ptr]),
    "pda_to_probs_batch_host": (C.c_int, [ptr, ptr, ptr, i64, i32]),
    "pda_association_workspace_bytes": (i64, [i64, i64, i64, i64, i32, i32, i32]),
    "pda_association_probs_batch": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, i64, i64, i64, i32, i32, i32, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_association_probs_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, i32]),
    "pda_association_perm_workspace_bytes": (i64, [i64, i64, i64, i64, i32, i32]),
    "pda_association_perm_probs_batch": (C.c_int, [ptr, ptr, ptr, ptr, ptr, i64, i64, i64, i64, i32, i32, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_association_perm_probs_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, i32]),
    "pda_association_probs_batch_host_multi": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, ptr, i32]),
    "pda_association_perm_probs_batch_host_multi": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, ptr, i32]),
    "pda_quadric_covs_batch": (C.c_int, [ptr, i64, ptr, ptr]),
    "pda_quadric_covs_batch_host": (C.c_int, [ptr, i64, ptr, i32]),
    "pda_quadric_cost_batch": (C.c_int, [ptr, ptr, ptr, ptr, ptr, ptr, i64, dbl, ptr, ptr, ptr, ptr, ptr]),
    "pda_quadric_cost_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, ptr, ptr, i64, dbl, ptr, i32]),
    "pda_association_from_moments_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, ptr, ptr, i64, dbl, i32, ptr, i32]),
    "pda_association_perm_from_moments_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, ptr, ptr, i64, dbl, ptr, ptr, i32]),
    "pda_association_from_moments_workspace_bytes": (i64, [i64, i32, i32, i64, i32]),
    "pda_association_from_moments_batch": (C.c_int, [ptr, ptr, ptr, i64, ptr, ptr, ptr, i64, i64, i32, i32, dbl, i32,
                                                     ptr, i64, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_association_perm_from_moments_workspace_bytes": (i64, [i64, i32, i32, i64]),
    "pda_association_perm_from_moments_batch": (C.c_int, [ptr, ptr, ptr, i64, ptr, ptr, ptr, i64, i64, i32, i32, dbl,
                                                          ptr, i64, ptr, ptr, ptr, i64, ptr]),
    "pda_asgn_bb_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, dbl, ptr, i32]),
    "pda_permanent_workspace_bytes": (i64, [i64]),
    "pda_permanent_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, ptr, i64, ptr]),
    "pda_permanent_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, i32]),
    "pda_permanent_range": (C.c_int, [ptr, i32, u64, u64, ptr, ptr, i64, ptr]),
    "pda_permanent_range_host": (C.c_int, [ptr, i32, u64, u64, ptr, i32]),
    "pda_permanent_batch_host_multi": (C.c_int, [ptr, ptr, ptr, ptr, i64, ptr, ptr, ptr, i32]),
    "pda_permanent_sharded_host": (C.c_int, [ptr, i32, ptr, i32, ptr]),
    "pda_permanent_approx_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, u64, ptr, ptr, ptr]),
    "pda_permanent_approx_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, u64, ptr, ptr, i32]),
    "pda_set_approx_seed": (None, [u64]),
    "pda_conditioned_permanent_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, i32]),
    "pda_permanent_prob_batch_host": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, ptr, i32]),
    "pda_permanent_prob_batch_host_multi": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, ptr, ptr, ptr, ptr, i32]),
    "pda_permanent_prob_workspace_bytes": (i64, [i64, i64, i64, i32, i32, i32]),
    "pda_permanent_prob_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, i64, i64, i32, i32, i32, ptr, ptr, ptr, ptr, i64, ptr]),
    "pda_conditioned_permanent_workspace_bytes": (i64, [i64, i32, i32]),
    "pda_conditioned_permanent_batch": (C.c_int, [ptr, ptr, ptr, ptr, i64, i32, i32, ptr, ptr, ptr, i64, ptr]),
}


class PdaError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libpda_b200 error {code}: {message}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(code: int) -> None:
    if code != 0:
        raise PdaError(int(code), lib().pda_last_error().decode(errors="replace"))
