"""B200-native Hull-White one-factor Monte Carlo engine (hot path of
giulialionetti/Monte-Carlo-simulation-of-Hull-White-model-and-sensitivities-computation).

The product is the CUDA library `lib/libhw1f.so` (C ABI in include/hw1f.h); this package is the
thin Python host layer over it.  There is no CPU fallback: importing works without a GPU, but
creating an Engine does not.
"""
from . import _ffi, engine, parallel
from ._ffi import LIB_PATH, BookVega, CapResult, Caplet, CashFlow, Params, Swaption, VegaResult, ZbcResult
from .engine import Engine, HW1FError, Rng, caplet_schedule, default_params, swaption_schedule

__all__ = ["engine", "parallel", "Engine", "Rng", "HW1FError", "default_params", "caplet_schedule", "swaption_schedule", "Params", "Caplet", "CapResult", "BookVega", "Swaption", "CashFlow", "ZbcResult", "VegaResult", "LIB_PATH", "_ffi"]
