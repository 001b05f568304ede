"""ctypes binding of the swaption book oracle (tests/swaption_oracle.c).

TEST INFRASTRUCTURE.  The shared library is compiled on first use, with the flags of oracle/Makefile, into the user's
temporary directory (keyed by a hash of its sources), so that the repository tree is never written to.  The moment
bound is cap_oracle.moment_bound: each P_j = A_j ex2(..) errs by at most eps relative (MUFU.EX2 vs exp2f), so with
c_j > 0 the coupon bond errs by |dBnd| <= eps Bnd and the payoff by |dx| <= eps y, the caplet's argument.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from cap_oracle import CFLAGS, ORACLE_DIR, moment_bound  # noqa: F401  (moment_bound: the bound of these moments)
from oracle_lib import OrcParams, Oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "swaption_oracle.c")] + [os.path.join(ORACLE_DIR, f) for f in
                                                        ("hw1f_oracle.c", "hw1f_oracle.h", "xorwow_ref.c", "xorwow_ref.h")]

SWAPTION_DTYPE = np.dtype([("T_exercise", np.float32), ("K", np.float32), ("N", np.float32), ("kind", np.int32),
                           ("step", np.int32), ("first_flow", np.int32), ("n_flows", np.int32), ("reserved", np.int32)])
FLOW_DTYPE = np.dtype([("T", np.float32), ("c", np.float32)])

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"hw1f_swaption_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"libhw1f_swaption_oracle_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-I", ORACLE_DIR, "-o", tmp, SOURCES[0], SOURCES[3], "-lm"],
                              stdout=subprocess.DEVNULL)
        os.replace(tmp, path)   # atomic: concurrent test processes see a complete library or none
    return path


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.orc_swaption_moments.argtypes = [C.POINTER(OrcParams), C.c_float, C.c_float, C.c_void_p, C.c_uint64,
                                              C.c_uint64, C.c_int64, C.c_uint64, C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def swaption_moments(oracle: Oracle, seed, n_pairs, swaptions, flows, P_mkt, f_mkt, first_path=0, offset=0, sigma=None):
    """moments[n + 1, 5] over antithetic pairs on the model of `oracle`; swaptions: any structured array with
    T_exercise, K, N, kind, first_flow, n_flows and optionally n_steps_exercise (< 0 or absent: the step nearest to
    T_exercise / dt); flows: any structured array with T and c"""
    sigma = oracle.p.sigma if sigma is None else sigma
    drift, _ = oracle.drift_tables(sigma)
    sw = np.zeros(len(swaptions), SWAPTION_DTYPE)
    for n in ("T_exercise", "K", "N", "kind", "first_flow", "n_flows"):
        sw[n] = swaptions[n]
    given = (swaptions["n_steps_exercise"] if "n_steps_exercise" in swaptions.dtype.names
             else np.full(len(swaptions), -1))
    dt = float(np.float32(oracle.dt))
    sw["step"] = [int(k) if k >= 0 else int(round(float(T) / dt)) for k, T in zip(given, sw["T_exercise"])]
    fl = np.zeros(len(flows), FLOW_DTYPE)
    fl["T"], fl["c"] = flows["T"], flows["c"]
    P_mkt = np.ascontiguousarray(P_mkt, np.float32)
    f_mkt = np.ascontiguousarray(f_mkt, np.float32)
    mom = np.zeros(5 * (len(sw) + 1), np.float64)
    lib().orc_swaption_moments(C.byref(oracle.p), sigma, oracle.sig_st(sigma), _p(drift), seed, first_path, n_pairs,
                               offset, _p(sw), len(sw), _p(fl), _p(P_mkt), _p(f_mkt), _p(mom))
    return mom.reshape(len(sw) + 1, 5)
