"""ctypes declarations of include/hw1f.h.  Loads <package>/lib/libhw1f.so and nothing else:
if the CUDA library is missing the import fails (there is no CPU path to fall back to)."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# HW1F_LIB selects an alternative build of the same library (kernel-variant experiments)
LIB_PATH = os.environ.get("HW1F_LIB") or os.path.join(HERE, "lib", "libhw1f.so")

OK = 0
MODE_REFERENCE_ORDER, MODE_DECOMPOSED = 0, 1
ASYNC_SLOTS = 4   # HW1F_ASYNC_SLOTS
ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE, ERR_UNSUPPORTED, ERR_NO_MODEL, ERR_COMM = 1, 2, 3, 4, 5, 6
KIND_CAP, KIND_FLOOR = 0, 1   # HW1F_KIND_*
MAX_CAPLETS = 100             # HW1F_MAX_CAPLETS
KIND_PAYER, KIND_RECEIVER = 0, 1   # HW1F_KIND_PAYER / HW1F_KIND_RECEIVER
MAX_SWAPTIONS = 100                # HW1F_MAX_SWAPTIONS
MAX_SWAPTION_FLOWS = 2048          # HW1F_MAX_SWAPTION_FLOWS


class Params(C.Structure):
    """hw1f_params (mirrors include/common.cuh:16-39 of the reference)."""
    _fields_ = [
        ("a", C.c_float), ("sigma", C.c_float), ("r0", C.c_float), ("T_final", C.c_float),
        ("n_steps", C.c_int32), ("n_mat", C.c_int32),
        ("theta_a0", C.c_float), ("theta_b0", C.c_float), ("theta_a1", C.c_float), ("theta_b1", C.c_float),
        ("theta_break", C.c_float), ("fd_theta_a1", C.c_float),
    ]


class Constants(C.Structure):
    _fields_ = [("dt", C.c_float), ("mat_spacing", C.c_float), ("exp_adt", C.c_float), ("sig_st", C.c_float),
                ("save_stride", C.c_int32)]


class ZbcResult(C.Structure):
    _fields_ = [
        ("mom", C.c_double * 5), ("n_total", C.c_uint64), ("n_steps_S1", C.c_int32), ("reserved", C.c_int32),
        ("mean_X", C.c_float), ("mean_Y", C.c_float), ("var_X", C.c_float), ("var_Y", C.c_float),
        ("cov", C.c_float), ("beta", C.c_float), ("control_adjustment", C.c_float),
        ("price_raw", C.c_float), ("price_cv", C.c_float), ("corr_single", C.c_float), ("corr", C.c_float),
        ("price_cv_f64", C.c_double), ("beta_f64", C.c_double), ("se_raw", C.c_double), ("se_cv", C.c_double),
        ("ci95_lo", C.c_double), ("ci95_hi", C.c_double),
        ("beta_se", C.c_double), ("corr_f64", C.c_double), ("corr_se", C.c_double),
    ]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n not in ("mom", "reserved")}
        d["mom"] = list(self.mom)
        return d


class VegaResult(C.Structure):
    _fields_ = [
        ("vega_pathwise", C.c_float), ("vega_pathwise_f64", C.c_double), ("vega_pathwise_se", C.c_double),
        ("price_minus", C.c_float), ("price_plus", C.c_float), ("vega_fd", C.c_float),
        ("price_minus_recal", C.c_float), ("price_plus_recal", C.c_float), ("vega_fd_recal", C.c_float),
        ("n_steps_S1", C.c_int32), ("ms_pathwise", C.c_float), ("ms_fd", C.c_float), ("ms_fd_recal", C.c_float),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class Caplet(C.Structure):
    """hw1f_caplet: one zero-coupon bond option of a cap (put) or floor (call) strip."""
    _fields_ = [("T_reset", C.c_float), ("T_pay", C.c_float), ("K", C.c_float), ("N", C.c_float),
                ("n_steps_reset", C.c_int32), ("reserved", C.c_int32)]


class CapResult(C.Structure):
    """hw1f_cap_result: one caplet, or the whole strip (moments over antithetic pairs)."""
    _fields_ = [("mom", C.c_double * 5), ("price_raw", C.c_double), ("se_raw", C.c_double),
                ("price_cv", C.c_double), ("se_cv", C.c_double), ("beta", C.c_double), ("corr", C.c_double),
                ("control_mean", C.c_double)]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "mom"}
        d["mom"] = list(self.mom)
        return d


class BookVega(C.Structure):
    """hw1f_book_vega: one option, or the whole book -- the sigma -/+ eps prices and the vega on common random numbers."""
    _fields_ = [("mom", C.c_double * 6), ("price_minus", C.c_double), ("se_minus", C.c_double),
                ("price_plus", C.c_double), ("se_plus", C.c_double), ("vega", C.c_double), ("vega_se", C.c_double)]

    def as_dict(self):
        d = {n: getattr(self, n) for n, _ in self._fields_ if n != "mom"}
        d["mom"] = list(self.mom)
        return d


class CashFlow(C.Structure):
    """hw1f_cash_flow: one payment (T, c) of a coupon bond."""
    _fields_ = [("T", C.c_float), ("c", C.c_float)]


class Swaption(C.Structure):
    """hw1f_swaption: an option on the coupon bond flows[first_flow, first_flow + n_flows), exercised at T_exercise."""
    _fields_ = [("T_exercise", C.c_float), ("K", C.c_float), ("N", C.c_float), ("kind", C.c_int32),
                ("n_steps_exercise", C.c_int32), ("first_flow", C.c_int32), ("n_flows", C.c_int32),
                ("reserved", C.c_int32)]


# every symbol include/hw1f.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_F = C.POINTER(C.c_float)
SYMBOLS = {
    "hw1f_abi_version": (C.c_int, []),
    "hw1f_status_string": (C.c_char_p, [C.c_int]),
    "hw1f_last_error": (C.c_char_p, [_P]),
    "hw1f_engine_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "hw1f_engine_destroy": (C.c_int, [_P]),
    "hw1f_engine_set_stream": (C.c_int, [_P, _P]),
    "hw1f_engine_device": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "hw1f_engine_set_mode": (C.c_int, [_P, C.c_int]),
    "hw1f_engine_get_mode": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "hw1f_engine_synchronize": (C.c_int, [_P]),
    "hw1f_default_params": (C.c_int, [C.POINTER(Params)]),
    "hw1f_set_model": (C.c_int, [_P, C.POINTER(Params)]),
    "hw1f_get_model": (C.c_int, [_P, C.POINTER(Params)]),
    "hw1f_get_constants": (C.c_int, [_P, C.POINTER(Constants)]),
    "hw1f_get_drift_table": (C.c_int, [_P, C.c_int, C.c_float, _P]),
    "hw1f_steps_to": (C.c_int, [_P, C.c_float, C.POINTER(C.c_int32)]),
    "hw1f_rng_create": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(_P)]),
    "hw1f_rng_clone": (C.c_int, [_P, C.POINTER(_P)]),
    "hw1f_rng_destroy": (C.c_int, [_P]),
    "hw1f_rng_tell": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    "hw1f_rng_seek": (C.c_int, [_P, C.c_uint64]),
    "hw1f_rng_info": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "hw1f_rng_prepare": (C.c_int, [_P, _P]),
    "hw1f_bond_curve": (C.c_int, [_P, _P, _P, _P, _P, _F]),
    "hw1f_bond_curve_submit": (C.c_int, [_P, _P, C.c_int32]),
    "hw1f_bond_curve_collect": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "hw1f_bond_curve_moments": (C.c_int, [_P, _P, _P]),
    "hw1f_bond_curve_finish": (C.c_int, [_P, _P, C.c_uint64, _P, _P, _P]),
    "hw1f_bond_curve_ci": (C.c_int, [_P, _P, _P, _P]),
    "hw1f_theta_calibrate": (C.c_int, [_P, _P, _P, _P, _P]),
    "hw1f_zbc_cv": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32, C.POINTER(ZbcResult), _F]),
    "hw1f_zbc_cv_moments": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32, _P]),
    "hw1f_zbc_cv_finish": (C.c_int, [_P, _P, C.c_uint64, C.c_float, C.POINTER(ZbcResult)]),
    "hw1f_zbc_cv_batch": (C.c_int, [_P, _P, C.c_int32, C.c_uint64, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32,
                                    C.POINTER(ZbcResult), _F]),
    "hw1f_vega_pathwise": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32,
                                     C.POINTER(VegaResult)]),
    "hw1f_vega_pathwise_moments": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32, _P]),
    "hw1f_vega_fd": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_float, C.c_int32,
                               C.POINTER(VegaResult)]),
    "hw1f_vega_fd_recalibrated": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32,
                                            C.POINTER(VegaResult)]),
    "hw1f_vega": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_float, C.c_int32,
                            C.POINTER(VegaResult)]),
    "hw1f_vega_pathwise_batch": (C.c_int, [_P, _P, C.c_int32, C.c_uint64, C.c_float, C.c_float, C.c_float, _P, _P,
                                           C.c_int32, _P, _F]),
    "hw1f_cap_floor": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.POINTER(CapResult), _F]),
    "hw1f_cap_floor_moments": (C.c_int, [_P, _P, C.c_int32, _P, C.c_int32, _P, _P, _P]),
    "hw1f_cap_floor_finish": (C.c_int, [_P, _P, C.c_uint64, _P, C.c_int32, _P, C.POINTER(CapResult)]),
    "hw1f_swaptions": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.POINTER(CapResult), _F]),
    "hw1f_swaptions_moments": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, _P]),
    "hw1f_swaptions_finish": (C.c_int, [_P, _P, C.c_uint64, _P, C.c_int32, _P, C.c_int32, _P, C.POINTER(CapResult)]),
    "hw1f_swaptions_vega": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.c_float, C.POINTER(CapResult),
                                      C.POINTER(BookVega), _F]),
    "hw1f_swaptions_vega_moments": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.c_int32, _P, _P, C.c_float, _P]),
    "hw1f_swaptions_vega_finish": (C.c_int, [_P, _P, C.c_uint64, _P, C.c_int32, _P, C.c_int32, _P, C.c_float,
                                             C.POINTER(CapResult), C.POINTER(BookVega)]),
    "hw1f_fused_moments": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32, _P]),
    "hw1f_fused_fd_moments": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_float, C.c_int32, _P]),
    "hw1f_fused": (C.c_int, [_P, _P, C.c_float, C.c_float, C.c_float, _P, _P, C.c_float, C.c_int32, _P, _P, _P,
                             C.POINTER(ZbcResult), C.POINTER(VegaResult), _F]),
    "hw1f_fused_finish": (C.c_int, [_P, _P, C.c_uint64, C.c_float, C.c_float, C.c_int32, _P, _P, _P,
                                    C.POINTER(ZbcResult), C.POINTER(VegaResult)]),
    "hw1f_multi_create": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "hw1f_multi_destroy": (C.c_int, [_P]),
    "hw1f_multi_device_count": (C.c_int, [_P, C.POINTER(C.c_int)]),
    "hw1f_multi_last_error": (C.c_char_p, [_P]),
    "hw1f_multi_set_model": (C.c_int, [_P, C.POINTER(Params)]),
    "hw1f_multi_set_mode": (C.c_int, [_P, C.c_int]),
    "hw1f_multi_bond_curve": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, _P, _P, _P, _F]),
    "hw1f_multi_zbc_cv": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float, C.c_float, C.c_float, _P, _P,
                                    C.c_int32, C.POINTER(ZbcResult)]),
    "hw1f_multi_fused": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float, C.c_float, C.c_float, _P, _P,
                                   C.c_float, C.c_int32, _P, _P, _P, C.POINTER(ZbcResult), C.POINTER(VegaResult), _F]),
    "hw1f_multi_vega_pathwise": (C.c_int, [_P, C.c_uint64, C.c_uint64, C.c_uint64, C.c_float, C.c_float, C.c_float, _P,
                                           _P, C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "hw1f_comm_create": (C.c_int, [_P, C.c_int, _P, C.POINTER(_P)]),
    "hw1f_comm_connect": (C.c_int, [_P, C.c_int, _P, _P]),
    "hw1f_comm_allreduce": (C.c_int, [_P, _P, C.c_int32]),
    "hw1f_comm_attach": (C.c_int, [_P, C.c_int]),
    "hw1f_comm_timeouts": (C.c_int, [_P, C.POINTER(C.c_uint32)]),
    "hw1f_comm_destroy": (C.c_int, [_P]),
    "hw1f_comm_last_error": (C.c_char_p, [_P]),
    "hw1f_sample_paths": (C.c_int, [_P, _P, C.c_int32, _P]),
    "hw1f_reduction_bench": (C.c_int, [_P, _P, C.c_int32, C.c_float, C.c_float, C.c_float, _P, _P, C.c_int32,
                                       C.c_int32, C.c_int32, _F, _F]),
    "hw1f_debug_rng": (C.c_int, [_P, _P, C.c_uint64, C.c_int32, _P, _P]),
    "hw1f_debug_normals": (C.c_int, [_P, _P, C.c_uint64, C.c_int32, _P]),
    "hw1f_host_rng_state": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, _P]),
    "hw1f_pipe_probe": (C.c_int, [_P, C.c_int32, C.c_int32, _F, C.POINTER(C.c_double)]),
    "hw1f_launch_count": (C.c_int, [_P, C.POINTER(C.c_uint64)]),
}

_lib = None


def load():
    """dlopen the engine.  Raises if the library has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "The HW1F engine is CUDA-only; there is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)   # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
