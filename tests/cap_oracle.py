"""ctypes binding of the cap / floor strip oracle (tests/cap_oracle.c).

TEST INFRASTRUCTURE.  The shared library is compiled on first use, with the flags of oracle/Makefile, into the user's
temporary directory (keyed by a hash of its sources), so that the repository tree is never written to.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle_lib import OrcParams, Oracle

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
SOURCES = [os.path.join(HERE, "cap_oracle.c")] + [os.path.join(ORACLE_DIR, f) for f in
                                                   ("hw1f_oracle.c", "hw1f_oracle.h", "xorwow_ref.c", "xorwow_ref.h")]
CFLAGS = ["-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-mavx2", "-mfma", "-fopenmp", "-Wall",
          "-Wextra"]

CAPLET_DTYPE = np.dtype([("T_reset", np.float32), ("T_pay", np.float32), ("K", np.float32), ("N", np.float32),
                         ("step", np.int32), ("reserved", np.int32)])

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"hw1f_cap_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"libhw1f_cap_oracle_{h.hexdigest()[:16]}.so")
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
        _lib.orc_cap_moments.argtypes = [C.POINTER(OrcParams), C.c_float, C.c_float, C.c_void_p, C.c_uint64,
                                         C.c_uint64, C.c_int64, C.c_uint64, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def moment_bound(ref, rel=3e-6, eps=2.4e-7):
    """Largest |engine - oracle| allowed per moment of cap_moments() (same [n + 1, 5] layout): `rel` relative, plus
    what MUFU.EX2 (the engine) vs exp2f (the oracle) may leave in the payoff.  P = A ex2(..) differs by up to eps
    relative, so x = D (K - P)^+ inherits an ABSOLUTE error |dx| <= eps y.  Summed over pairs that gives eps sY for
    sum X, and 2 x dx + dx^2 <= 2 eps x y + eps^2 y^2 for sum X^2 (the square term matters only when every pair of a
    tiny run is at the money and the oracle's x is zero), eps sYY for sum XY.  The controls get no slack."""
    sX, sY, sXX, sYY, sXY = np.asarray(ref).T
    slack = np.stack([eps * sY, 0 * sY, 2 * eps * sXY + eps * eps * sYY, 0 * sY, eps * sYY], axis=1)
    return rel * np.abs(ref) + slack


def cap_moments(oracle: Oracle, seed, n_pairs, caplets, P_mkt, f_mkt, kind="cap", first_path=0, offset=0, sigma=None):
    """moments[n + 1, 5] over antithetic pairs on the model of `oracle`; caplets: any structured array with T_reset,
    T_pay, K, N and optionally n_steps_reset (< 0 or absent: the step nearest to T_reset / dt)"""
    sigma = oracle.p.sigma if sigma is None else sigma
    drift, _ = oracle.drift_tables(sigma)
    caps = np.zeros(len(caplets), CAPLET_DTYPE)
    for n in ("T_reset", "T_pay", "K", "N"):
        caps[n] = caplets[n]
    given = caplets["n_steps_reset"] if "n_steps_reset" in caplets.dtype.names else np.full(len(caplets), -1)
    dt = float(np.float32(oracle.dt))
    caps["step"] = [int(k) if k >= 0 else int(round(float(T) / dt)) for k, T in zip(given, caps["T_reset"])]
    P_mkt = np.ascontiguousarray(P_mkt, np.float32)
    f_mkt = np.ascontiguousarray(f_mkt, np.float32)
    mom = np.zeros(5 * (len(caps) + 1), np.float64)
    lib().orc_cap_moments(C.byref(oracle.p), sigma, oracle.sig_st(sigma), _p(drift), seed, first_path, n_pairs, offset,
                          0 if kind == "cap" else 1, _p(caps), len(caps), _p(P_mkt), _p(f_mkt), _p(mom))
    return mom.reshape(len(caps) + 1, 5)
