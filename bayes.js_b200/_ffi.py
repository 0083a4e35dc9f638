"""ctypes binding of include/amwg.h (libamwg_b200.so).

There is no CPU fallback: if the shared object is missing or no CUDA device is usable, every entry
point raises.  The library is looked up in-tree (bayes.js_b200/libamwg_b200.so); build it with
``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C bayes.js_b200/csrc``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libamwg_b200.so")

# ---- opcodes / plate kinds: keep in sync with include/amwg.h (checked by tests/test_abi.py) ----
_OPS = """END CONST COMP DATA DATA_I COMP_I ADD SUB MUL DIV NEG LOG EXP SQRT ABS POW LT LE GT GE EQ NE AND OR NOT SELECT
LGAMMA LFACTORIAL LCHOOSE LBETA LD_NORM LD_UNIF LD_BETA LD_BERN LD_POIS LD_CAUCHY LD_LAPLACE LD_GAMMA LD_INVGAMMA
LD_LNORM LD_PARETO LD_T LD_WEIBULL LD_LOGIS LD_EXP LD_BINOM LD_NBINOM LD_HYPER ACC PLATE STORE LOOP_BEGIN LOOP_END
NORM_K UNIF_K BETA_K ACC_RANGE PLATE_SS NORM_SS CACHED CAND""".split()
OP = {name: i for i, name in enumerate(_OPS)}
OP_COUNT = len(_OPS)
PLATE_GENERIC, PLATE_NORM_IID, PLATE_BERN_IID, PLATE_NORM_GROUPED, PLATE_POIS_LOGLIN = range(5)
REAL, INT, BINARY = 0, 1, 2
ABI_VERSION = 8


class AmwgParam(C.Structure):
    _fields_ = [("type", C.c_int32), ("n_comp", C.c_int32), ("dim0", C.c_int32), ("comp_offset", C.c_int32),
                ("lower", C.c_double), ("upper", C.c_double)]


class AmwgCompOptions(C.Structure):
    _fields_ = [("prop_log_scale", C.c_double), ("batch_size", C.c_double), ("max_adaptation", C.c_double),
                ("initial_adaptation", C.c_double), ("target_accept_rate", C.c_double),
                ("is_adapting", C.c_int32), ("_pad", C.c_int32)]


class AmwgColumn(C.Structure):
    _fields_ = [("values", C.POINTER(C.c_double)), ("n", C.c_int64)]


class AmwgPlate(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n", C.c_int32), ("col", C.c_int32 * 4), ("iparam", C.c_int32 * 4)]


class AmwgModel(C.Structure):
    _fields_ = [("abi_version", C.c_int32),
                ("n_params", C.c_int32), ("params", C.POINTER(AmwgParam)),
                ("n_comp", C.c_int32), ("init", C.POINTER(C.c_double)),
                ("comp_options", C.POINTER(AmwgCompOptions)),
                ("n_code", C.c_int32), ("code", C.POINTER(C.c_int32)),
                ("logpost_prog", C.c_int32), ("derived_prog", C.c_int32), ("n_derived", C.c_int32),
                ("n_consts", C.c_int32), ("consts", C.POINTER(C.c_double)),
                ("n_columns", C.c_int32), ("columns", C.POINTER(AmwgColumn)),
                ("n_plates", C.c_int32), ("plates", C.POINTER(AmwgPlate)),
                ("n_fold", C.c_int32), ("fold_prog", C.POINTER(C.c_int32)), ("fold_dst", C.POINTER(C.c_int32)),
                ("n_terms", C.c_int32), ("comp_prog", C.POINTER(C.c_int32)),
                ("touch_off", C.POINTER(C.c_int32)), ("touch_terms", C.POINTER(C.c_int32)),
                ("n_block_params", C.c_int32), ("block_params", C.POINTER(C.c_int32)), ("term_block_comp", C.POINTER(C.c_int32)),
                ("stat_prog", C.c_int32), ("n_sum_terms", C.c_int32),
                ("n_variant_comps", C.c_int32), ("variant_comps", C.POINTER(C.c_int32)),
                ("variant_logpost", C.POINTER(C.c_int32)), ("variant_derived", C.POINTER(C.c_int32))]


EXPORTS = ["amwg_create", "amwg_destroy", "amwg_burn", "amwg_sample", "amwg_sample_device", "amwg_get_state", "amwg_get_log_post",
           "amwg_set_adapting", "amwg_info", "amwg_kernel_launches", "amwg_last_sweep_kernel_ms", "amwg_n_chains",
           "amwg_last_error", "amwg_abi_version", "amwg_ld_eval", "amwg_primitive_eval",
           "amwg_summary_moments", "amwg_summary_digit_hist", "amwg_summary_autocov", "amwg_summary_rank_keys", "amwg_summary_rank_sort",
           "amwg_summary_rank_runs", "amwg_summary_rank_z", "amwg_summary_rank_scatter", "amwg_peak_fp64", "amwg_jit_status", "amwg_jit_compile_check"]

_lib = None


class AmwgError(RuntimeError):
    """Raised when the native library is missing or a call fails (no CPU fallback exists)."""


def lib():
    """Load libamwg_b200.so once and declare the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AmwgError(f"{LIB_PATH} not found: build it (make -C bayes.js_b200/csrc). "
                        "The sampler has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
    pd, pi = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    L.amwg_create.argtypes = [C.POINTER(AmwgModel), u64, u64, u64, C.c_int, C.POINTER(vp)]
    L.amwg_create.restype = C.c_int
    L.amwg_destroy.argtypes = [vp]; L.amwg_destroy.restype = None
    L.amwg_burn.argtypes = [vp, i64]; L.amwg_burn.restype = C.c_int
    L.amwg_sample.argtypes = [vp, i64, i64, pi, i32, vp]; L.amwg_sample.restype = C.c_int
    L.amwg_sample_device.argtypes = [vp, i64, i64, pi, i32, vp]; L.amwg_sample_device.restype = C.c_int
    L.amwg_get_state.argtypes = [vp, vp]; L.amwg_get_state.restype = C.c_int
    L.amwg_get_log_post.argtypes = [vp, vp]; L.amwg_get_log_post.restype = C.c_int
    L.amwg_set_adapting.argtypes = [vp, i32]; L.amwg_set_adapting.restype = C.c_int
    L.amwg_info.argtypes = [vp, vp, vp, vp]; L.amwg_info.restype = C.c_int
    L.amwg_kernel_launches.argtypes = [vp]; L.amwg_kernel_launches.restype = i64
    L.amwg_last_sweep_kernel_ms.argtypes = [vp]; L.amwg_last_sweep_kernel_ms.restype = dbl
    L.amwg_n_chains.argtypes = [vp]; L.amwg_n_chains.restype = u64
    L.amwg_last_error.argtypes = []; L.amwg_last_error.restype = C.c_char_p
    L.amwg_abi_version.argtypes = []; L.amwg_abi_version.restype = C.c_int
    L.amwg_ld_eval.argtypes = [i32, vp, i32, i64, vp, C.c_int]; L.amwg_ld_eval.restype = C.c_int
    L.amwg_primitive_eval.argtypes = [i32, vp, i64, u64, u64, vp, C.c_int]; L.amwg_primitive_eval.restype = C.c_int
    L.amwg_summary_moments.argtypes = [C.c_int, vp, i64, i32, i64, vp]; L.amwg_summary_moments.restype = C.c_int
    L.amwg_summary_digit_hist.argtypes = [C.c_int, vp, i64, i32, i64, i32, vp, i32, vp]; L.amwg_summary_digit_hist.restype = C.c_int
    L.amwg_summary_autocov.argtypes = [C.c_int, vp, i64, i32, i64, vp, vp, i32, i32, i32, vp]; L.amwg_summary_autocov.restype = C.c_int
    L.amwg_summary_rank_keys.argtypes = [C.c_int, vp, i64, i32, i64, i32, vp, vp, vp]; L.amwg_summary_rank_keys.restype = C.c_int
    L.amwg_summary_rank_sort.argtypes = [C.c_int, vp, vp, i64, vp, vp, vp]; L.amwg_summary_rank_sort.restype = C.c_int
    L.amwg_summary_rank_runs.argtypes = [C.c_int, vp, vp, vp, vp, i64, vp, vp, vp, vp]; L.amwg_summary_rank_runs.restype = C.c_int
    L.amwg_summary_rank_z.argtypes = [C.c_int, vp, i64, i64, i64, vp]; L.amwg_summary_rank_z.restype = C.c_int
    L.amwg_summary_rank_scatter.argtypes = [C.c_int, vp, vp, i64, vp, vp, i32, i64, i32]; L.amwg_summary_rank_scatter.restype = C.c_int
    L.amwg_jit_status.argtypes = [vp, C.c_char_p, i64]; L.amwg_jit_status.restype = C.c_int
    L.amwg_jit_compile_check.argtypes = [C.POINTER(AmwgModel), u64, C.c_char_p, i64, C.c_char_p, i64]; L.amwg_jit_compile_check.restype = C.c_int
    L.amwg_peak_fp64.argtypes = [C.c_int, C.c_int, pd, pd]; L.amwg_peak_fp64.restype = C.c_int
    if L.amwg_abi_version() != ABI_VERSION:
        raise AmwgError("libamwg_b200.so ABI version mismatch")
    _lib = L
    return L


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().amwg_last_error().decode("utf-8", "replace")
        raise AmwgError(msg or what or "amwg call failed")
