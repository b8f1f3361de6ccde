"""
ctypes mirror of include/rvlnl.h and the loader of the in-tree librvlnl.so.

There is no CPU fallback: if the CUDA library is missing the import of any compute entry point
raises, loudly.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_int32, c_int64, c_uint64,
                    c_void_p)

RVL_ABI_VERSION = 1
RVL_MAX_PLANETS = 8
RVL_MAX_INST = 16
RVL_MAX_LINPAR = 8
RVL_MAX_DIM = 128
RVL_MAX_PEERS = 16

RVL_ECC_DIRECT, RVL_ECC_SECOS_SESIN, RVL_ECC_ECOS_ESIN = 0, 1, 2
RVL_PHASE_MA0, RVL_PHASE_ML0 = 0, 1

(RVL_PRIOR_UNIFORM, RVL_PRIOR_JEFFREYS, RVL_PRIOR_MODJEFFREYS, RVL_PRIOR_UNIFORMFREQ,
 RVL_PRIOR_TRUNCRAYLEIGH, RVL_PRIOR_NORMAL, RVL_PRIOR_LOGNORMAL, RVL_PRIOR_TABLE) = range(8)

RVL_ERRORS = {0: "OK", -1: "EINVAL", -2: "ENODEV", -3: "ECUDA", -4: "ESTATE", -5: "ENOMEM",
              -6: "EPEER"}


class rvl_param(Structure):
    _fields_ = [("slot", c_int32), ("reserved", c_int32), ("value", c_double)]


class rvl_planet_desc(Structure):
    _fields_ = [("amp", rvl_param), ("period", rvl_param), ("e1", rvl_param),
                ("e2", rvl_param), ("phase", rvl_param), ("epoch", rvl_param),
                ("amp_is_log", c_int32), ("period_is_log", c_int32),
                ("ecc_mode", c_int32), ("phase_mode", c_int32)]


class rvl_model_desc(Structure):
    _fields_ = [("abi_version", c_int32), ("ndim", c_int32), ("n_planets", c_int32),
                ("n_inst", c_int32), ("jitter_in_model", c_int32),
                ("drift_in_model", c_int32), ("n_linpar", c_int32), ("itmax", c_int32),
                ("tol", c_double), ("tref", c_double),
                ("planet", rvl_planet_desc * RVL_MAX_PLANETS),
                ("offset", rvl_param * RVL_MAX_INST), ("jitter", rvl_param * RVL_MAX_INST),
                ("drift", rvl_param * 4), ("linpar", rvl_param * RVL_MAX_LINPAR)]


class rvl_prior_desc(Structure):
    _fields_ = [("kind", c_int32), ("table_len", c_int32), ("table_offset", c_int64),
                ("p", c_double * 4)]


class rvl_counters_t(Structure):
    _fields_ = [("n_points", c_uint64), ("n_solves", c_uint64),
                ("n_newton_iters", c_uint64), ("n_cap_hits", c_uint64),
                ("n_invalid", c_uint64)]


class rvl_slice_args(Structure):
    _fields_ = ([("k", c_int32), ("d", c_int32), ("n_out", c_int32), ("m", c_int32),
                 ("seed", c_uint64), ("move", ctypes.c_uint32), ("shrink_round", ctypes.c_uint32)] +
                [(n, c_uint64) for n in ("lmin", "chol", "u", "theta", "lcur", "dirn", "lo", "hi", "lo2",
                                         "hi2", "tval", "pending", "cand_out", "inside_out", "ll_out",
                                         "cand", "inside", "cand_ll", "cand_th", "stats")])


class rvl_slice_runs(Structure):
    _fields_ = ([("n_runs", c_int32), ("reserved", c_int32)] +
                [(n, c_uint64) for n in ("run_of", "walker_of", "seeds", "lmin", "chol", "stats")])


class rvl_slice_live(Structure):
    _fields_ = ([("nlive", c_int32), ("d", c_int32), ("round", ctypes.c_uint32),
                 ("reserved", ctypes.c_uint32)] +
                [(n, c_uint64) for n in ("u_live", "th_live", "l_live", "order", "kk", "start", "lstart")])


_dp = POINTER(c_double)

# name -> (restype, argtypes); every symbol include/rvlnl.h declares
SYMBOLS = {
    "rvl_abi_version": (c_int32, []),
    "rvl_create": (c_int32, [POINTER(c_void_p), c_int32]),
    "rvl_create_multi": (c_int32, [POINTER(c_void_p), POINTER(c_int32), c_int32]),
    "rvl_device_count": (c_int32, [c_void_p, POINTER(c_int32)]),
    "rvl_destroy": (None, [c_void_p]),
    "rvl_reset": (c_int32, [c_void_p]),
    "rvl_last_error": (c_char_p, [c_void_p]),
    "rvl_set_data": (c_int32, [c_void_p, _dp, _dp, _dp, POINTER(c_int32), c_int32, c_int32]),
    "rvl_set_linpar": (c_int32, [c_void_p, c_int32, _dp, c_int32]),
    "rvl_set_model": (c_int32, [c_void_p, POINTER(rvl_model_desc)]),
    "rvl_set_priors": (c_int32, [c_void_p, POINTER(rvl_prior_desc), c_int32, _dp, c_int64]),
    "rvl_set_option": (c_int32, [c_void_p, c_char_p, c_int64]),
    # hot host-buffer calls: plain addresses (c_void_p takes an int or any ctypes pointer), so that
    # the Python wrappers can pass ndarray.ctypes.data without building pointer objects
    "rvl_transform": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p]),
    "rvl_loglike": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p]),
    "rvl_transform_loglike": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "rvl_transform_dev": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "rvl_loglike_dev": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "rvl_loglike_dev_scatter": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_uint64),
                                          c_int32, c_int64, c_void_p]),
    "rvl_loglike_dev_gather": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_uint64),
                                         c_int32, c_int32, c_int64, c_int64, c_uint64, c_void_p]),
    "rvl_loglike_gather": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, POINTER(c_uint64),
                                     c_int32, c_int32, c_int64, c_uint64]),
    "rvl_gather_status": (c_int32, [c_void_p]),
    "rvl_host_register": (c_int32, [c_void_p, c_int64, POINTER(c_uint64)]),
    "rvl_host_unregister": (c_int32, [c_void_p]),
    "rvl_loglike_scatter_host": (c_int32, [c_void_p, c_void_p, c_int64, c_uint64, c_int64, c_int64,
                                           c_int32, c_uint64]),
    "rvl_wait_host_flags": (c_int32, [c_void_p, c_int32, c_uint64, c_int32]),
    "rvl_transform_loglike_dev": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                            c_void_p]),
    "rvl_trueanomaly": (c_int32, [c_void_p, _dp, c_int32, c_double, _dp, c_int32, c_double]),
    "rvl_kepler_rv": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, ctypes.c_uint32,
                                c_void_p, c_void_p, POINTER(c_uint64)]),
    "rvl_kepler_rv_dev": (c_int32, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, ctypes.c_uint32,
                                    c_void_p, c_void_p, c_void_p, c_void_p]),
    "rvl_counters": (c_int32, [c_void_p, POINTER(rvl_counters_t)]),
    "rvl_reset_counters": (c_int32, [c_void_p]),
    "rvl_last_kernel_ms": (c_int32, [c_void_p, _dp]),
    "rvl_last_gather_wait_ms": (c_int32, [c_void_p, _dp]),
    "rvl_launch_count": (c_int32, [c_void_p, POINTER(c_uint64)]),
    "rvl_fp64_peak": (c_int32, [c_void_p, _dp]),
    "rvl_device_info": (c_int32, [c_void_p, POINTER(c_int32), POINTER(c_int32),
                                  POINTER(c_int32)]),
    "rvl_read_trace": (c_int32, [c_void_p, POINTER(c_uint64), c_int32, POINTER(c_int32)]),
    "rvl_fip_accumulate": (c_int32, [c_int32, _dp, _dp, c_int32, _dp, c_int32, _dp, c_int64, c_double,
                                     c_int32, c_double, c_double, _dp, _dp]),
    "rvl_fip_last_error": (c_char_p, []),
    "rvl_order_planets": (c_int32, [c_int32, _dp, c_int64, c_int32, POINTER(c_int32), POINTER(c_int32),
                                    c_int32, c_int32, _dp, _dp]),
    "rvl_order_last_error": (c_char_p, []),
    "rvl_post_release": (None, []),
    "rvl_slice_phase": (c_int32, [c_int32, POINTER(rvl_slice_args), c_void_p]),
    "rvl_slice_phase_wrapped": (c_int32, [c_int32, POINTER(rvl_slice_args), POINTER(ctypes.c_uint32),
                                          c_void_p]),
    "rvl_slice_phase_runs": (c_int32, [c_int32, POINTER(rvl_slice_args), POINTER(rvl_slice_runs),
                                       POINTER(ctypes.c_uint32), c_void_p]),
    "rvl_slice_runs_init": (c_int32, [POINTER(rvl_slice_runs), POINTER(rvl_slice_live), c_void_p]),
    "rvl_slice_runs_whiten": (c_int32, [POINTER(rvl_slice_runs), POINTER(rvl_slice_live),
                                        POINTER(ctypes.c_uint32), c_void_p]),
    "rvl_slice_runs_starts": (c_int32, [POINTER(rvl_slice_args), POINTER(rvl_slice_runs),
                                        POINTER(rvl_slice_live), c_void_p]),
    "rvl_slice_last_error": (c_char_p, []),
    "rvl_plan_describe": (c_int32, [POINTER(c_int32), c_int64, POINTER(c_int64), c_int32]),
}

# RVL_LIB: another build of the same library (kernel A/B experiments, tools/build_variants.py);
# it must export the same ABI -- there is still no fallback of any kind
LIB_PATH = os.environ.get("RVL_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)),
                                                      "librvlnl.so")

_lib = None


def load():
    """Load librvlnl.so (built in-tree by ``evidence_b200.build``) and bind its symbols."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA library first "
                "(python -c 'import __graft_entry__ as g; g.build()').  "
                "evidence_b200 has no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        if lib.rvl_abi_version() != RVL_ABI_VERSION:
            raise ImportError("librvlnl.so ABI version mismatch; rebuild")
        _lib = lib
    return _lib
