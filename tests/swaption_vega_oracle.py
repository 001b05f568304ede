"""ctypes binding of the book vega oracle (tests/swaption_vega_oracle.c), and the bounds of its comparison with the engine.

TEST INFRASTRUCTURE.  The shared library is compiled on first use, with the flags of oracle/Makefile, into the user's
temporary directory (keyed by a hash of its sources), so that the repository tree is never written to.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from cap_oracle import CFLAGS, ORACLE_DIR, moment_bound
from oracle_lib import OrcParams, Oracle
from swaption_oracle import FLOW_DTYPE, SWAPTION_DTYPE

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "swaption_vega_oracle.c")] + [os.path.join(ORACLE_DIR, f) for f in
                                                             ("hw1f_oracle.c", "hw1f_oracle.h", "xorwow_ref.c",
                                                              "xorwow_ref.h")]

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"hw1f_swaption_vega_oracle_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"libhw1f_swaption_vega_oracle_{h.hexdigest()[:16]}.so")
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
        _lib.orc_swaption_vega_moments.argtypes = [C.POINTER(OrcParams), C.c_float, C.c_uint64, C.c_uint64, C.c_int64,
                                                   C.c_uint64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p]
        _lib.orc_vega_set_threads.argtypes = [C.c_int]
    return _lib


def set_threads(n):
    """OpenMP threads of the oracles in this process (they share one OpenMP runtime)"""
    lib().orc_vega_set_threads(int(n))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def vega_moments(oracle: Oracle, seed, n_pairs, swaptions, flows, P_mkt, f_mkt, eps, first_path=0, offset=0):
    """(mom[11 (n + 1)] in the engine's layout, aux[2, n + 1, 5]) on the model of `oracle`; swaptions, flows as
    swaption_oracle.swaption_moments takes them.  aux: X, Y, X^2, Y^2, XY of the sigma - eps and sigma + eps scenarios."""
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
    n = len(sw)
    mom = np.zeros(11 * (n + 1), np.float64)
    aux = np.zeros(10 * (n + 1), np.float64)
    lib().orc_swaption_vega_moments(C.byref(oracle.p), eps, seed, first_path, n_pairs, offset, _p(sw), n, _p(fl),
                                    _p(P_mkt), _p(f_mkt), _p(mom), _p(aux))
    return mom, aux.reshape(2, n + 1, 5)


def split(mom, n):
    """the engine's 11 (n + 1) vector as (base[n + 1, 5], vega[n + 1, 6])"""
    mom = np.asarray(mom)
    return mom[:5 * (n + 1)].reshape(n + 1, 5), mom[5 * (n + 1):].reshape(n + 1, 6)


def vega_bound(vega_ref, aux, rel=3e-6, eps=2.4e-7):
    """Largest |engine - oracle| allowed per entry of the [n + 1, 6] vega block.  Sum X_s and sum X_s^2 get
    moment_bound of scenario s (aux[s] holds its X, Y moments).  Per pair the payoff may differ by
    |dX_s| <= rel X_s + eps Y_s (X_s, Y_s >= 0; the book's too, as sums over the options), so
    sum D gets the sum of the two sum-X bounds, and with E = 2 sum (dX_+^2 + dX_-^2) <= 4 sum_s (rel^2 X_s^2 + eps^2 Y_s^2)
    (a bound on sum dD^2), sum D^2 gets 2 sqrt(sum D^2 E) + E (Cauchy-Schwarz)."""
    bm, bp = moment_bound(aux[0], rel=rel, eps=eps), moment_bound(aux[1], rel=rel, eps=eps)
    E = 4 * sum(rel * rel * a[:, 2] + eps * eps * a[:, 3] for a in aux)
    sDD = np.abs(vega_ref[:, 5])
    return np.stack([bm[:, 0], bm[:, 2], bp[:, 0], bp[:, 2], bm[:, 0] + bp[:, 0], 2 * np.sqrt(sDD * E) + E], axis=1)


def vega_algebra(v, n_pairs, eps):
    """hw1f_book_vega's statistics from six pair moments"""
    n = float(n_pairs)

    def mean_se(s, ss):
        sx, sxx = 0.5 * s, 0.25 * ss
        mx = sx / n
        return mx, np.sqrt(max((sxx - sx * mx) / (n - 1), 0.0) / n)
    pm, sm = mean_se(v[0], v[1])
    pp, sp = mean_se(v[2], v[3])
    d, sd = mean_se(v[4], v[5])
    return {"price_minus": pm, "se_minus": sm, "price_plus": pp, "se_plus": sp, "vega": d / (2 * eps),
            "vega_se": sd / (2 * eps)}
