"""ctypes binding of libpyperiod_b200.so (include/pyperiod_b200.h).

There is no CPU fallback: if the shared object is missing the import of any product
class raises, telling the user to run `python -m pyperiod_b200.build`.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PYPERIOD_B200_LIB selects an alternative build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("PYPERIOD_B200_LIB") or os.path.join(HERE, "libpyperiod_b200.so")

ABI_VERSION = 10

METRIC_NORM, METRIC_GAMMA, METRIC_MAXABS, METRIC_IMPOSED = 0, 1, 2, 3
STATUS_OK, STATUS_NO_PERIOD, STATUS_OVERFLOW, STATUS_SINGULAR, STATUS_GUARD = 0, 1, 2, 3, 4
STATUS_TOO_LARGE, STATUS_ZERO_INPUT = 5, 6
BASIS_NATURAL, BASIS_RAMANUJAN = 0, 1
RAM_FP64, RAM_TF32, RAM_F32COMPAT = 0, 1, 2
STAGING_AUTO, STAGING_SHARED, STAGING_GLOBAL = 0, 1, 2
ALGO_SWEEP, ALGO_MBEST, ALGO_S2L, ALGO_BCORR, ALGO_QO, ALGO_RAMANUJAN = 0, 1, 2, 3, 4, 5
ALGO_PROJECT, ALGO_BFREQ = 6, 7
QO_KIND_FIND, QO_KIND_SOLVE, QO_KIND_MURESAN, QO_KIND_SOLVE_RAMANUJAN = 0, 1, 2, 3

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64
_f64 = C.c_double
_sz = C.c_size_t

# name -> (restype, argtypes); every symbol include/pyperiod_b200.h declares
SIGNATURES = {
    "pp_abi_version": (C.c_int, []),
    "pp_last_error": (C.c_char_p, []),
    "pp_sweep_passes": (C.c_int, [_i32, _i32, _i32, _i32]),
    "pp_device_info": (C.c_int, [_p, _p, _p, _p, _p]),
    "pp_grid_size": (C.c_int, [_i32, _i32, _i32, _i32]),
    "pp_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32]),
    "pp_project": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _p, _i64, _i32, _p]),
    "pp_periodic_norm": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p]),
    "pp_sweep": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p, _p, _sz,
                           _p]),
    "pp_mbest": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _i32,
                           _p, _p, _p, _p, _p, _p, _p, _sz, _p, _p]),
    "pp_small_to_large": (C.c_int, [_p, _i64, _i32, _i32, _f64, _i32, _i32, _i32, _p, _p, _i32, _i32,
                                    _p, _p, _p, _p, _p, _p, _sz, _p]),
    "pp_best_correlation": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _f64, _i32, _i32, _i32, _p, _p, _i32,
                                      _p, _p, _p, _p, _p, _sz, _p]),
    "pp_best_frequency_round": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p, _i32, _i32,
                                          _p, _p]),
    "pp_muresan_powers": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _p, _p, _p, _p]),
    "pp_comm_load": (C.c_int, [C.c_char_p]),
    "pp_comm_version": (C.c_int, []),
    "pp_comm_unique_id": (C.c_int, [_p]),
    "pp_comm_init": (C.c_int, [_p, _i32, _i32, _p]),
    "pp_comm_destroy": (C.c_int, [_p]),
    "pp_gather": (C.c_int, [_p, _p, _p, _sz, _i32, _p]),
    "pp_microbench": (C.c_int, [_i32, _i32, _p]),
    "pp_ramanujan_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32]),
    "pp_ramanujan_norms": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _p, _sz, _p]),
    "pp_ramanujan_norms_tf32": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _p, _sz, _p]),
    "pp_ramanujan_norms_f32compat": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _p, _sz,
                                              _p]),
    "pp_ramanujan_select": (C.c_int, [_p, _i32, _i32, _i32, _f64, _i32, _p, _p, _p]),
    "pp_ramanujan_fits_on_chip": (C.c_int, [_i32, _i32, _i32, _i32, _i32]),
    "pp_long_ramanujan_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "pp_long_ramanujan_norms": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _i32, _p, _sz, _p]),
    "pp_ramanujan_divisor_fits_on_chip": (C.c_int, [_i32, _i32, _i32, _i32]),
    "pp_ramanujan_divisor_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32]),
    "pp_ramanujan_norms_divisor": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _p, _sz,
                                             _p]),
    "pp_qo_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i32]),
    "pp_qo_find_periods": (C.c_int, [_p, _i64, _i32, _i32, _i32, _f64, _i32, _i32, _i32, _i32, _i32, _i32, _p, _i32, _i32,
                                     _p, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _i32, _p, _p, _sz, _p,
                                     _p]),
    "pp_qo_solve": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _i32, _p, _i32,
                              _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "pp_qo_solve_ramanujan": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _i32, _p, _i32,
                                        _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "pp_qo_get_periods": (C.c_int, [_i32, _i32, _i32, _i32, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _p, _p]),
    "pp_qo_dictionary_rows": (C.c_int, [_i32, _i32, _p, _p, _i32, _p, _i32, _p, _p]),
    "pp_fits_on_chip": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "pp_long_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i32]),
    "pp_long_project": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _p, _i64, _i32, _p, _sz, _p]),
    "pp_long_sweep": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p, _p, _sz,
                                _p]),
    "pp_long_mbest": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _i32,
                                _p, _p, _p, _p, _p, _p, _p, _sz, _p]),
    "pp_long_small_to_large": (C.c_int, [_p, _i64, _i32, _i32, _f64, _i32, _i32, _i32, _p, _p, _i32, _i32,
                                         _p, _p, _p, _p, _p, _p, _sz, _p]),
    "pp_long_best_correlation": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _f64, _i32, _i32, _p, _p, _i32,
                                           _p, _p, _p, _p, _p, _sz, _p]),
    "pp_long_best_frequency_round": (C.c_int, [_p, _i32, _i32, _p, _i32, _i32, _i32, _i32, _p, _p, _i32, _p, _p, _p,
                                               _i32, _i32, _p, _p, _sz, _p]),
    "pp_qo_solve_rows": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _i32, _i32, _i32, _p, _p, _i64, _p, _p, _p,
                                   _sz, _p]),
    "pp_qo_fits_on_chip": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32]),
    "pp_long_qo_max_rows": (_i32, [_i32]),
    "pp_long_qo_workspace_bytes": (_sz, [_i32, _i32, _i32, _i32, _i32, _i32, _i32, _sz]),
    "pp_long_qo_find_periods": (C.c_int, [_p, _i64, _i32, _i32, _i32, _f64, _i32, _i32, _i32, _i32, _i32, _p, _i32,
                                          _i32, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _p, _p, _p, _sz, _p]),
    "pp_long_qo_solve": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _i32, _p, _i32,
                                   _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "pp_long_qo_solve_ramanujan": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _i32, _i32, _p, _i32, _i32, _p, _i32,
                                             _p, _p, _p, _p, _p, _i64, _p, _p, _p, _p, _sz, _p]),
    "pp_long_qo_solve_rows": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _i32, _i32, _i32, _p, _p, _i64, _p, _p,
                                        _p, _sz, _p]),
    "pp_long_muresan_powers": (C.c_int, [_p, _i64, _i32, _i32, _i32, _i32, _p, _i32, _p, _p, _p, _p, _sz, _p]),
}

_lib = None


class PPError(RuntimeError):
    pass


def load():
    """Load the library once and attach signatures.  Raises if it was never built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA library is not built and there is no CPU path. "
            "Run `python -m pyperiod_b200.build` (needs nvcc).")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    got = lib.pp_abi_version()
    if got != ABI_VERSION:
        raise ImportError(f"libpyperiod_b200.so ABI {got} != expected {ABI_VERSION}; rebuild it")
    _lib = lib
    return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().pp_last_error().decode("utf-8", "replace")
        raise PPError(f"{what} failed ({rc}): {msg}")


FOLD_HIERARCHICAL, FOLD_DIRECT, FOLD_HIERARCHICAL_NO_RIDERS, FOLD_NOMINATE_F32 = 0, 1, 2, 3


FOLD_NAMES = {"hierarchical": FOLD_HIERARCHICAL, "direct": FOLD_DIRECT, "no_riders": FOLD_HIERARCHICAL_NO_RIDERS,
              "f32": FOLD_NOMINATE_F32}

# The C library keeps no process-wide state: the fold mode and the optional profile buffer are arguments of every
# call.  These two module variables are only the DEFAULTS the Python classes pass when an instance does not set
# its own (`Periods(..., fold_mode=...)`); tests and the tuning tools use them to switch whole scripts.
_default_fold_mode = FOLD_HIERARCHICAL
_profile_ptr = 0


def set_fold_mode(mode: int):
    """Default fold mode of instances that do not choose one (FOLD_*; see include/pyperiod_b200.h)."""
    global _default_fold_mode
    if int(mode) not in FOLD_NAMES.values():
        raise PPError("unknown fold mode")
    _default_fold_mode = int(mode)


def default_fold_mode() -> int:
    return _default_fold_mode


def resolve_fold_mode(mode) -> int:
    """None -> the module default; a FOLD_* value or one of FOLD_NAMES."""
    if mode is None:
        return _default_fold_mode
    if isinstance(mode, str):
        return FOLD_NAMES[mode]
    return int(mode)


def set_profile_buffer(tensor_or_none):
    """Device buffer of 8 uint64 the M-best / QO kernels add phase cycle counts to (development aid)."""
    global _profile_ptr
    _profile_ptr = 0 if tensor_or_none is None else int(tensor_or_none.data_ptr())


def profile_ptr() -> C.c_void_p:
    return C.c_void_p(_profile_ptr)


def sweep_passes(n: int, pmin: int, pmax: int, fold_mode=None) -> int:
    """Passes over a window of n samples per ranking sweep under `fold_mode` (default: the module default)."""
    return int(load().pp_sweep_passes(int(n), int(pmin), int(pmax), resolve_fold_mode(fold_mode)))


def microbench(kind: int, iters: int = 4000) -> dict:
    """Measured chip-wide peak: kind 0 = shared-memory bytes/s, kind 1 = FP64 adds/s, kind 2 = DMMA flop/s."""
    out = (C.c_double * 3)()
    check(load().pp_microbench(kind, iters, out), "pp_microbench")
    return {"per_s": out[0], "sm_mhz": out[1], "ms": out[2]}


def fits_on_chip(algo: int, n: int, pmax: int, num: int, metric: int, trunc: int, orth: int, fold_mode: int,
                 smem_bytes: int) -> bool:
    """Whether the on-chip plan of a call fits `smem_bytes` of shared memory per block (pp_fits_on_chip; no device
    is touched).  Calls whose plan does not fit run on the global-memory path (pp_long_*)."""
    rc = load().pp_fits_on_chip(int(algo), int(n), int(pmax), int(num), int(metric), int(trunc), int(orth),
                                int(fold_mode), int(smem_bytes))
    if rc < 0:
        check(rc, "pp_fits_on_chip")
    return rc == 1


def qo_fits_on_chip(kind: int, n: int, pmax: int, num: int, rmax: int, basis: int, fold_mode: int,
                    smem_bytes: int) -> bool:
    """Whether the on-chip QO / Muresan launch `kind` (QO_KIND_*) fits `smem_bytes` of shared memory per block
    (pp_qo_fits_on_chip; no device is touched).  Launches that do not fit run on the global-memory path."""
    rc = load().pp_qo_fits_on_chip(int(kind), int(n), int(pmax), int(num), int(rmax), int(basis), int(fold_mode),
                                   int(smem_bytes))
    if rc < 0:
        check(rc, "pp_qo_fits_on_chip")
    return rc == 1


def ramanujan_fits_on_chip(mode: int, n: int, qmin: int, qmax: int, smem_bytes: int) -> bool:
    """Whether the on-chip Ramanujan periodogram of `mode` (RAM_*) fits `smem_bytes` of shared memory per block
    (pp_ramanujan_fits_on_chip; no device is touched).  fp64 calls that do not fit run on the global-memory path."""
    rc = load().pp_ramanujan_fits_on_chip(int(mode), int(n), int(qmin), int(qmax), int(smem_bytes))
    if rc < 0:
        check(rc, "pp_ramanujan_fits_on_chip")
    return rc == 1


def ramanujan_divisor_fits_on_chip(n: int, qmin: int, qmax: int, smem_bytes: int) -> bool:
    """Whether the on-chip divisor-form Ramanujan periodogram fits `smem_bytes` of shared memory per block
    (pp_ramanujan_divisor_fits_on_chip; no device is touched).  Calls that do not fit run from global memory."""
    rc = load().pp_ramanujan_divisor_fits_on_chip(int(n), int(qmin), int(qmax), int(smem_bytes))
    if rc < 0:
        check(rc, "pp_ramanujan_divisor_fits_on_chip")
    return rc == 1


def long_qo_max_rows(smem_bytes: int) -> int:
    """Rows of the largest dictionary the global-memory QO path solves with `smem_bytes` of shared memory."""
    return int(load().pp_long_qo_max_rows(int(smem_bytes)))


def device_info() -> dict:
    lib = load()
    vals = [C.c_int32() for _ in range(5)]
    check(lib.pp_device_info(*[C.byref(v) for v in vals]), "pp_device_info")
    keys = ["sm_count", "smem_optin_bytes", "cc_major", "cc_minor", "clock_khz"]
    return {k: v.value for k, v in zip(keys, vals)}
