"""Host-side mirror of the reference's operator surface, on top of the C ABI (include/hw1f.h).

The reference is four single-file CUDA drivers; each method below names the driver code it stands
for.  Everything heavy happens in libhw1f.so on the GPU; this file only marshals numpy arrays.
"""
import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import BookVega, CapResult, Caplet, CashFlow, Constants, Params, Swaption, VegaResult, ZbcResult


class HW1FError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"hw1f status {status}: {message}")
        self.status = status


def default_params(**overrides):
    """H_* constants and N_* macros of include/common.cuh:16-39."""
    p = Params()
    _ffi.load().hw1f_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(k)
        setattr(p, k, v)
    return p


def _f32(a, n=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if n is not None and a.size != n:
        raise ValueError(f"expected {n} float32 values, got {a.size}")
    return a


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


# numpy mirror of hw1f_caplet
CAPLET_DTYPE = np.dtype([(n, np.float32 if t is C.c_float else np.int32) for n, t in Caplet._fields_])
assert CAPLET_DTYPE.itemsize == C.sizeof(Caplet)


def caplet_schedule(resets, pays, strike_rate, notional=1.0):
    """Caplets on the simple rates L(T_r, T_p) struck at `strike_rate` (scalar or one per caplet), as the bond options
    the engine prices: a caplet pays M tau (L - kappa)^+ at T_p, which is worth N ZBP(T_r, T_p, K) with tau = T_p - T_r,
    K = 1 / (1 + tau kappa) and N = M (1 + tau kappa) (a floorlet: N ZBC).  Reset steps are left to the engine
    (n_steps_reset = -1: the step nearest to T_r / dt).  Returns a structured array of hw1f_caplet; no GPU needed."""
    resets = np.atleast_1d(np.asarray(resets, np.float64))
    pays = np.atleast_1d(np.asarray(pays, np.float64))
    if resets.shape != pays.shape:
        raise ValueError("resets and pays must have the same length")
    kappa = np.broadcast_to(np.asarray(strike_rate, np.float64), resets.shape)
    M = np.broadcast_to(np.asarray(notional, np.float64), resets.shape)
    tau = pays - resets
    grow = 1.0 + tau * kappa
    out = np.zeros(resets.shape, CAPLET_DTYPE)
    out["T_reset"], out["T_pay"] = resets, pays
    out["K"], out["N"] = 1.0 / grow, M * grow
    out["n_steps_reset"] = -1
    return out


def _caplets(caplets):
    """structured array of hw1f_caplet (caplet_schedule), a ctypes Caplet array, or a sequence of Caplet / dicts"""
    if isinstance(caplets, np.ndarray) and caplets.dtype.names:
        a = np.zeros(caplets.shape, CAPLET_DTYPE)
        for n in CAPLET_DTYPE.names:
            if n in caplets.dtype.names:
                a[n] = caplets[n]
            elif n == "n_steps_reset":
                a[n] = -1
        return np.ascontiguousarray(a.ravel())
    rows = []
    for c in caplets:
        if isinstance(c, Caplet):
            rows.append(tuple(getattr(c, n) for n in CAPLET_DTYPE.names))
        else:
            rows.append((c["T_reset"], c["T_pay"], c["K"], c["N"], c.get("n_steps_reset", -1), 0))
    return np.array(rows, CAPLET_DTYPE)


def _kind(kind):
    if kind in ("cap", _ffi.KIND_CAP):
        return _ffi.KIND_CAP
    if kind in ("floor", _ffi.KIND_FLOOR):
        return _ffi.KIND_FLOOR
    return int(kind) if isinstance(kind, (int, np.integer)) else -1   # the engine rejects it with a message


def _cap_results(res, n):
    """per-caplet numpy arrays and the strip as a dict"""
    rows = [res[i].as_dict() for i in range(n)]
    out = {k: np.array([r[k] for r in rows], np.float64)
           for k in ("price_cv", "se_cv", "price_raw", "se_raw", "beta", "corr", "control_mean")}
    out["mom"] = np.array([r["mom"] for r in rows], np.float64).reshape(n, 5)
    out["strip"] = res[n].as_dict()
    return out


# numpy mirrors of hw1f_swaption and hw1f_cash_flow
SWAPTION_DTYPE = np.dtype([(n, np.float32 if t is C.c_float else np.int32) for n, t in Swaption._fields_])
CASH_FLOW_DTYPE = np.dtype([(n, np.float32) for n, _ in CashFlow._fields_])
assert SWAPTION_DTYPE.itemsize == C.sizeof(Swaption) and CASH_FLOW_DTYPE.itemsize == C.sizeof(CashFlow)


def _swaption_kind(kind):
    if kind in ("payer", _ffi.KIND_PAYER):
        return _ffi.KIND_PAYER
    if kind in ("receiver", _ffi.KIND_RECEIVER):
        return _ffi.KIND_RECEIVER
    return int(kind) if isinstance(kind, (int, np.integer)) else -1   # the engine rejects it with a message


def swaption_schedule(expiries, tenors, strike_rate, freq=1, notional=1.0, kind="payer"):
    """European swaptions on spot-starting swaps, one per (expiry, tenor) pair (the arguments broadcast against each
    other; a grid is expiries and tenors repeated to its cells), as the coupon-bond options the engine prices.  The
    swap from T_e to T_e + tenor pays the fixed rate kappa every 1 / freq years, so the option is on the bond with flows
    c = kappa / freq at T_e + k / freq (the last c += 1), strike K = 1 and multiplier N = M (notional); a payer
    swaption is a put on that bond, a receiver swaption a call.  Exercise steps are left to the engine
    (n_steps_exercise = -1: the step nearest to T_e / dt).  Returns (swaptions, flows), structured arrays of
    hw1f_swaption and hw1f_cash_flow; no GPU needed."""
    kinds = np.asarray(kind, dtype=object)
    Te, ten, kappa, M, kd = np.broadcast_arrays(np.asarray(expiries, np.float64), np.asarray(tenors, np.float64),
                                                np.asarray(strike_rate, np.float64), np.asarray(notional, np.float64),
                                                kinds)
    Te, ten, kappa, M, kd = (np.atleast_1d(a).ravel() for a in (Te, ten, kappa, M, kd))
    n_cpn = np.rint(ten * freq).astype(np.int64)
    if (n_cpn < 1).any() or (np.abs(ten * freq - n_cpn) > 1e-9).any():
        raise ValueError("every tenor must be a positive whole number of coupon periods (tenor * freq)")
    sw = np.zeros(len(Te), SWAPTION_DTYPE)
    fl = np.zeros(int(n_cpn.sum()), CASH_FLOW_DTYPE)
    row = 0
    for i in range(len(Te)):
        k = np.arange(1, n_cpn[i] + 1)
        c = np.full(n_cpn[i], kappa[i] / freq)
        c[-1] += 1.0
        fl["T"][row:row + n_cpn[i]] = Te[i] + k / freq
        fl["c"][row:row + n_cpn[i]] = c
        sw[i] = (Te[i], 1.0, M[i], _swaption_kind(kd[i]), -1, row, n_cpn[i], 0)
        row += n_cpn[i]
    return sw, fl


def _swaption_book(swaptions, flows):
    """structured arrays (swaption_schedule) or sequences of tuples in the field order of hw1f_swaption /
    hw1f_cash_flow -> contiguous arrays of the ABI structs"""
    def conv(x, dt, defaults):
        if isinstance(x, np.ndarray) and x.dtype.names:
            a = np.zeros(x.shape, dt)
            for n in dt.names:
                if n in x.dtype.names:
                    a[n] = x[n]
                elif n in defaults:
                    a[n] = defaults[n]
            return np.ascontiguousarray(a.ravel())
        return np.array([tuple(r) for r in x], dt)
    return conv(swaptions, SWAPTION_DTYPE, {"n_steps_exercise": -1}), conv(flows, CASH_FLOW_DTYPE, {})


def _book_results(res, n):
    out = _cap_results(res, n)
    out["book"] = out.pop("strip")
    return out


def _add_vega(out, vres, n, book_key):
    """the hw1f_book_vega rows into a result dict: per-option arrays, and the book's values into out[book_key]"""
    rows = [vres[i].as_dict() for i in range(n)]
    for k in ("price_minus", "se_minus", "price_plus", "se_plus", "vega", "vega_se"):
        out[k] = np.array([r[k] for r in rows], np.float64)
    out["vega_mom"] = np.array([r["mom"] for r in rows], np.float64).reshape(n, 6)
    book = vres[n].as_dict()
    book["vega_mom"] = book.pop("mom")
    out[book_key].update(book)
    return out


def _caplet_book(caplets, kind):
    """a strip of caplets as a book of one-flow options: flow (T_pay, 1), payer for a cap (a put on the bond), receiver
    for a floor (a call), exercised at the reset step"""
    cap = _caplets(caplets)
    k = _kind(kind)
    sw = np.zeros(len(cap), SWAPTION_DTYPE)
    sw["T_exercise"], sw["K"], sw["N"] = cap["T_reset"], cap["K"], cap["N"]
    sw["kind"] = {_ffi.KIND_CAP: _ffi.KIND_PAYER, _ffi.KIND_FLOOR: _ffi.KIND_RECEIVER}.get(k, -1)
    sw["n_steps_exercise"] = cap["n_steps_reset"]
    sw["first_flow"] = np.arange(len(cap))
    sw["n_flows"] = 1
    fl = np.zeros(len(cap), CASH_FLOW_DTYPE)
    fl["T"], fl["c"] = cap["T_pay"], 1.0
    return sw, fl


class Rng:
    """(seed, first_path, n_paths, normal offset): replaces the curandState array + init_rng
    (include/common.cuh:277-280) and the state backup/restore copies of src/3:407-435."""

    def __init__(self, seed, n_paths, first_path=0, _handle=None):
        self._lib = _ffi.load()
        if _handle is None:
            h = C.c_void_p()
            st = self._lib.hw1f_rng_create(int(seed) & (2 ** 64 - 1), int(first_path), int(n_paths), C.byref(h))
            if st != _ffi.OK:
                raise HW1FError(st, "hw1f_rng_create")
            _handle = h
        self._h = _handle

    def clone(self):
        h = C.c_void_p()
        st = self._lib.hw1f_rng_clone(self._h, C.byref(h))
        if st != _ffi.OK:
            raise HW1FError(st, "hw1f_rng_clone")
        return Rng(0, 1, _handle=h)

    def tell(self):
        off = C.c_uint64()
        self._lib.hw1f_rng_tell(self._h, C.byref(off))
        return off.value

    def seek(self, offset):
        self._lib.hw1f_rng_seek(self._h, int(offset))
        return self

    @property
    def info(self):
        s, f, n = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self._lib.hw1f_rng_info(self._h, C.byref(s), C.byref(f), C.byref(n))
        return {"seed": s.value, "first_path": f.value, "n_paths": n.value}

    @property
    def n_paths(self):
        return self.info["n_paths"]

    def __del__(self):
        try:
            if self._h:
                self._lib.hw1f_rng_destroy(self._h)
                self._h = None
        except Exception:
            pass


def host_rng_state(seed, path, normal_offset=0):
    """XORWOW words {d, v0..v4} from the engine's HOST jump algebra (no GPU involved)."""
    out = np.zeros(6, np.uint32)
    st = _ffi.load().hw1f_host_rng_state(int(seed) & (2 ** 64 - 1), int(path), int(normal_offset), _ptr(out))
    if st != _ffi.OK:
        raise HW1FError(st, "hw1f_host_rng_state")
    return out


class Engine:
    """One engine per process and GPU (the reference: one process, one GPU, default stream)."""

    K_DEFAULT = float(np.exp(np.float32(-0.1)).astype(np.float32))  # K = expf(-0.1f), src/2:110

    def __init__(self, device=0, params=None, stream=None):
        self._lib = _ffi.load()
        h = C.c_void_p()
        st = self._lib.hw1f_engine_create(int(device), C.byref(h))
        if st != _ffi.OK:
            raise HW1FError(st, self._lib.hw1f_status_string(st).decode() +
                            " (the HW1F engine needs a B200-class CUDA device; there is no CPU fallback)")
        self._h = h
        if stream is not None:
            self.set_stream(stream)
        self.set_model(params if params is not None else default_params())

    # -- plumbing --
    def _check(self, st):
        if st != _ffi.OK:
            raise HW1FError(st, self._lib.hw1f_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.hw1f_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream):
        """cuda_stream: integer cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream) or None."""
        self._check(self._lib.hw1f_engine_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    def set_mode(self, mode):
        """_ffi.MODE_REFERENCE_ORDER (per-path reference float sequence) or _ffi.MODE_DECOMPOSED (default)"""
        self._check(self._lib.hw1f_engine_set_mode(self._h, int(mode)))

    @property
    def mode(self):
        m = C.c_int()
        self._lib.hw1f_engine_get_mode(self._h, C.byref(m))
        return m.value

    def synchronize(self):
        self._check(self._lib.hw1f_engine_synchronize(self._h))

    @property
    def launch_count(self):
        n = C.c_uint64()
        self._lib.hw1f_launch_count(self._h, C.byref(n))
        return n.value

    # -- model (compute_constants / compute_drift_tables, common.cuh:60-110) --
    def set_model(self, params):
        self._check(self._lib.hw1f_set_model(self._h, C.byref(params)))
        raw = bytes(params)
        if raw != getattr(self, "_params_raw", None):      # derived constants only change with the parameters
            c = Constants()
            self._check(self._lib.hw1f_get_constants(self._h, C.byref(c)))
            self.constants = c
            self.n_mat, self.n_steps = params.n_mat, params.n_steps
            self._params_raw = raw
        self.params = params

    def drift_table(self, which=0, sigma=None):
        out = np.zeros(self.n_steps, np.float32)
        self._check(self._lib.hw1f_get_drift_table(self._h, which, self.params.sigma if sigma is None else sigma,
                                                   _ptr(out)))
        return out

    def steps_to(self, S1):
        n = C.c_int32()
        self._check(self._lib.hw1f_steps_to(self._h, S1, C.byref(n)))
        return n.value

    # -- Q1: simulate_zcb + compute_average_and_forward (src/1_bond_pricing.cu:65-79) --
    def bond_curve(self, rng, with_se=True, timing=True):
        """timing=False: no CUDA events around the simulation (sim_ms is None)"""
        P = np.zeros(self.n_mat, np.float32)
        f = np.zeros(self.n_mat, np.float32)
        se = np.zeros(self.n_mat, np.float32) if with_se else None
        ms = C.c_float()
        self._check(self._lib.hw1f_bond_curve(self._h, rng._h, _ptr(P), _ptr(f), _ptr(se) if with_se else None,
                                              C.byref(ms) if timing else None))
        return {"P": P, "f": f, "P_se": se, "sim_ms": ms.value if timing else None}

    def bond_curve_submit(self, rng, slot=0):
        """hw1f_bond_curve in two halves: enqueue everything now, read the slot later (up to ASYNC_SLOTS in flight)"""
        self._check(self._lib.hw1f_bond_curve_submit(self._h, rng._h, int(slot)))

    def bond_curve_collect(self, slot=0, with_se=True):
        P = np.zeros(self.n_mat, np.float32)
        f = np.zeros(self.n_mat, np.float32)
        se = np.zeros(self.n_mat, np.float32) if with_se else None
        self._check(self._lib.hw1f_bond_curve_collect(self._h, int(slot), _ptr(P), _ptr(f), _ptr(se) if with_se else None))
        return {"P": P, "f": f, "P_se": se}

    def bond_curve_moments(self, rng, d_moments_ptr):
        """async: device pointer to 2*n_mat doubles (e.g. a torch.float64 CUDA tensor's data_ptr())."""
        self._check(self._lib.hw1f_bond_curve_moments(self._h, rng._h, C.c_void_p(d_moments_ptr)))

    def bond_curve_finish(self, d_moments_ptr, n_paths_total, with_se=True):
        P = np.zeros(self.n_mat, np.float32)
        f = np.zeros(self.n_mat, np.float32)
        se = np.zeros(self.n_mat, np.float32) if with_se else None
        self._check(self._lib.hw1f_bond_curve_finish(self._h, C.c_void_p(d_moments_ptr), int(n_paths_total), _ptr(P),
                                                     _ptr(f), _ptr(se) if with_se else None))
        return {"P": P, "f": f, "P_se": se}

    def bond_curve_ci(self):
        """standard errors of f(0,T), theta(T) (and P, by batch means) for the last bond-curve launch on this engine"""
        f_se, th_se, p_se = (np.zeros(self.n_mat, np.float32) for _ in range(3))
        self._check(self._lib.hw1f_bond_curve_ci(self._h, _ptr(f_se), _ptr(th_se), _ptr(p_se)))
        return {"f_se": f_se, "theta_se": th_se, "P_se_batch": p_se}

    # -- Q2a: recover_theta (src/2_option_pricing.cu:14-35,70-102) --
    def theta_calibrate(self, f):
        f = _f32(f, self.n_mat)
        rec, ref, T = (np.zeros(self.n_mat, np.float32) for _ in range(3))
        self._check(self._lib.hw1f_theta_calibrate(self._h, _ptr(f), _ptr(rec), _ptr(ref), _ptr(T)))
        # print_theta_comparison (src/2:39-68): statistics over every SAVE_STRIDE-th maturity only
        idx = np.arange(0, self.n_mat, self.constants.save_stride)
        err = np.abs(rec[idx] - ref[idx]).astype(np.float32)
        return {"theta_rec": rec, "theta_ref": ref, "T": T, "max_error": float(err.max()),
                "mean_error": float(err.astype(np.float32).sum(dtype=np.float32) / np.float32(len(idx))),
                "success": bool(err.max() < 0.01)}

    # -- Q2b: run_ZBC_control_variate (src/2:107-208) --
    def zbc_cv(self, rng, P_mkt, f_mkt, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res, ms = ZbcResult(), C.c_float()
        self._check(self._lib.hw1f_zbc_cv(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K, _ptr(P_mkt),
                                          _ptr(f_mkt), n_steps_S1, C.byref(res), C.byref(ms)))
        d = res.as_dict()
        d["sim_ms"] = ms.value
        return d

    def zbc_cv_moments(self, rng, P_mkt, f_mkt, d_moments_ptr, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        self._check(self._lib.hw1f_zbc_cv_moments(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K,
                                                  _ptr(P_mkt), _ptr(f_mkt), n_steps_S1, C.c_void_p(d_moments_ptr)))

    def zbc_cv_finish(self, d_moments_ptr, n_paths_total, P0S2):
        res = ZbcResult()
        self._check(self._lib.hw1f_zbc_cv_finish(self._h, C.c_void_p(d_moments_ptr), int(n_paths_total), P0S2,
                                                 C.byref(res)))
        return res.as_dict()

    # run_zbc_statistical_validation (src/2:210-302): all runs in one launch
    def zbc_cv_batch(self, seeds, n_paths, P_mkt, f_mkt, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
        res = (ZbcResult * len(seeds))()
        ms = C.c_float()
        self._check(self._lib.hw1f_zbc_cv_batch(self._h, _ptr(seeds), len(seeds), int(n_paths), S1, S2,
                                                self.K_DEFAULT if K is None else K, _ptr(P_mkt), _ptr(f_mkt),
                                                n_steps_S1, res, C.byref(ms)))
        return [r.as_dict() for r in res], ms.value

    # -- caps and floors: every caplet of a strip in one simulation pass (no reference call site) --
    def cap_floor(self, rng, caplets, P_mkt, f_mkt, kind="cap"):
        """kind "cap" (bond puts) or "floor" (bond calls); caplets as from caplet_schedule().  Per-caplet arrays
        price_cv, se_cv, price_raw, se_raw, beta, corr, control_mean, mom[n, 5], the whole strip under "strip"."""
        cap = _caplets(caplets)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res, ms = (CapResult * (len(cap) + 1))(), C.c_float()
        self._check(self._lib.hw1f_cap_floor(self._h, rng._h, _kind(kind), _ptr(cap), len(cap), _ptr(P_mkt), _ptr(f_mkt),
                                             res, C.byref(ms)))
        out = _cap_results(res, len(cap))
        out["sim_ms"] = ms.value
        return out

    def cap_floor_moments(self, rng, caplets, P_mkt, f_mkt, d_moments_ptr, kind="cap"):
        """async: device pointer to 5 * (len(caplets) + 1) doubles"""
        cap = _caplets(caplets)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        self._check(self._lib.hw1f_cap_floor_moments(self._h, rng._h, _kind(kind), _ptr(cap), len(cap), _ptr(P_mkt),
                                                     _ptr(f_mkt), C.c_void_p(d_moments_ptr)))

    def cap_floor_finish(self, d_moments_ptr, n_paths_total, caplets, P_mkt):
        cap = _caplets(caplets)
        P_mkt = _f32(P_mkt, self.n_mat)
        res = (CapResult * (len(cap) + 1))()
        self._check(self._lib.hw1f_cap_floor_finish(self._h, C.c_void_p(d_moments_ptr), int(n_paths_total), _ptr(cap),
                                                    len(cap), _ptr(P_mkt), res))
        return _cap_results(res, len(cap))

    # -- European swaptions: a book of coupon-bond options in one simulation pass (no reference call site) --
    def swaptions(self, rng, swaptions, flows, P_mkt, f_mkt):
        """swaptions, flows as from swaption_schedule().  Per-option arrays price_cv, se_cv, price_raw, se_raw, beta,
        corr, control_mean, mom[n, 5], the whole book under "book", and sim_ms."""
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res, ms = (CapResult * (len(sw) + 1))(), C.c_float()
        self._check(self._lib.hw1f_swaptions(self._h, rng._h, _ptr(sw), len(sw), _ptr(fl), len(fl), _ptr(P_mkt),
                                             _ptr(f_mkt), res, C.byref(ms)))
        out = _book_results(res, len(sw))
        out["sim_ms"] = ms.value
        return out

    def swaptions_moments(self, rng, swaptions, flows, P_mkt, f_mkt, d_moments_ptr):
        """async: device pointer to 5 * (len(swaptions) + 1) doubles"""
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        self._check(self._lib.hw1f_swaptions_moments(self._h, rng._h, _ptr(sw), len(sw), _ptr(fl), len(fl),
                                                     _ptr(P_mkt), _ptr(f_mkt), C.c_void_p(d_moments_ptr)))

    def swaptions_finish(self, d_moments_ptr, n_paths_total, swaptions, flows, P_mkt):
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt = _f32(P_mkt, self.n_mat)
        res = (CapResult * (len(sw) + 1))()
        self._check(self._lib.hw1f_swaptions_finish(self._h, C.c_void_p(d_moments_ptr), int(n_paths_total), _ptr(sw),
                                                    len(sw), _ptr(fl), len(fl), _ptr(P_mkt), res))
        return _book_results(res, len(sw))

    # -- vega of a swaption book / cap strip: sigma -/+ eps on common random numbers (no reference call site) --
    def swaptions_vega(self, rng, swaptions, flows, P_mkt, f_mkt, eps=1e-3):
        """What swaptions() returns (bit-identical), plus per-option arrays price_minus, se_minus, price_plus, se_plus
        (raw prices of the models with sigma -/+ eps, which keep the curve), vega, vega_se and vega_mom[n, 6]; the
        book's values under "book", and sim_ms."""
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res, vres, ms = (CapResult * (len(sw) + 1))(), (BookVega * (len(sw) + 1))(), C.c_float()
        self._check(self._lib.hw1f_swaptions_vega(self._h, rng._h, _ptr(sw), len(sw), _ptr(fl), len(fl), _ptr(P_mkt),
                                                  _ptr(f_mkt), float(eps), res, vres, C.byref(ms)))
        out = _add_vega(_book_results(res, len(sw)), vres, len(sw), "book")
        out["sim_ms"] = ms.value
        return out

    def swaptions_vega_moments(self, rng, swaptions, flows, P_mkt, f_mkt, d_moments_ptr, eps=1e-3):
        """async: device pointer to 11 * (len(swaptions) + 1) doubles (the swaptions_moments vector first)"""
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        self._check(self._lib.hw1f_swaptions_vega_moments(self._h, rng._h, _ptr(sw), len(sw), _ptr(fl), len(fl),
                                                          _ptr(P_mkt), _ptr(f_mkt), float(eps),
                                                          C.c_void_p(d_moments_ptr)))

    def swaptions_vega_finish(self, d_moments_ptr, n_paths_total, swaptions, flows, P_mkt, eps=1e-3):
        sw, fl = _swaption_book(swaptions, flows)
        P_mkt = _f32(P_mkt, self.n_mat)
        res, vres = (CapResult * (len(sw) + 1))(), (BookVega * (len(sw) + 1))()
        self._check(self._lib.hw1f_swaptions_vega_finish(self._h, C.c_void_p(d_moments_ptr), int(n_paths_total),
                                                         _ptr(sw), len(sw), _ptr(fl), len(fl), _ptr(P_mkt), float(eps),
                                                         res, vres))
        return _add_vega(_book_results(res, len(sw)), vres, len(sw), "book")

    def cap_floor_vega(self, rng, caplets, P_mkt, f_mkt, kind="cap", eps=1e-3):
        """What cap_floor() returns (the strip under "strip"), plus the vega arrays of swaptions_vega(): the strip is
        priced as the book of its one-flow options (a one-flow option performs the caplet's float operations)."""
        sw, fl = _caplet_book(caplets, kind)
        out = self.swaptions_vega(rng, sw, fl, P_mkt, f_mkt, eps=eps)
        out["strip"] = out.pop("book")
        return out

    # -- Q3 (src/3_sensitivity_analysis.cu) --
    def vega_pathwise(self, rng, P_mkt, f_mkt, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res = VegaResult()
        self._check(self._lib.hw1f_vega_pathwise(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K,
                                                 _ptr(P_mkt), _ptr(f_mkt), n_steps_S1, C.byref(res)))
        return res.as_dict()

    def vega_pathwise_moments(self, rng, P_mkt, f_mkt, d_moments_ptr, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        self._check(self._lib.hw1f_vega_pathwise_moments(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K,
                                                         _ptr(P_mkt), _ptr(f_mkt), n_steps_S1,
                                                         C.c_void_p(d_moments_ptr)))

    def vega_fd(self, rng, P_mkt, f_mkt, eps=0.001, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res = VegaResult()
        self._check(self._lib.hw1f_vega_fd(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K, _ptr(P_mkt),
                                           _ptr(f_mkt), eps, n_steps_S1, C.byref(res)))
        return res.as_dict()

    def vega_fd_recalibrated(self, rng, eps=0.001, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        res = VegaResult()
        self._check(self._lib.hw1f_vega_fd_recalibrated(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K,
                                                        eps, n_steps_S1, C.byref(res)))
        return res.as_dict()

    def vega(self, rng, P_mkt, f_mkt, eps=0.001, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        """main() of src/3 with the reference's draw windows (SURVEY 3.3)."""
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        res = VegaResult()
        self._check(self._lib.hw1f_vega(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K, _ptr(P_mkt),
                                        _ptr(f_mkt), eps, n_steps_S1, C.byref(res)))
        return res.as_dict()

    def vega_pathwise_batch(self, seeds, n_paths, P_mkt, f_mkt, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        seeds = np.ascontiguousarray(np.asarray(seeds, dtype=np.uint64))
        vega = np.zeros(len(seeds), np.float32)
        ms = C.c_float()
        self._check(self._lib.hw1f_vega_pathwise_batch(self._h, _ptr(seeds), len(seeds), int(n_paths), S1, S2,
                                                       self.K_DEFAULT if K is None else K, _ptr(P_mkt), _ptr(f_mkt),
                                                       n_steps_S1, _ptr(vega), C.byref(ms)))
        return vega, ms.value

    # -- fused single-window pass: curve + ZBC/CV + pathwise vega + CRN FD bumps in ONE launch --
    def fused(self, rng, P_mkt, f_mkt, eps=0.001, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        P, f, se = (np.zeros(self.n_mat, np.float32) for _ in range(3))
        z, v, ms = ZbcResult(), VegaResult(), C.c_float()
        self._check(self._lib.hw1f_fused(self._h, rng._h, S1, S2, self.K_DEFAULT if K is None else K, _ptr(P_mkt),
                                         _ptr(f_mkt), eps, n_steps_S1, _ptr(P), _ptr(f), _ptr(se), C.byref(z),
                                         C.byref(v), C.byref(ms)))
        return {"P": P, "f": f, "P_se": se, "zbc": z.as_dict(), "vega": v.as_dict(), "sim_ms": ms.value}

    def fused_moments(self, rng, P_mkt, f_mkt, d_moments_ptr, eps=None, S1=5.0, S2=10.0, K=None, n_steps_S1=-1):
        """async; eps=None: 2*n_mat+8 doubles, eps given: 2*n_mat+18 (FD bumps ride along)"""
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        K = self.K_DEFAULT if K is None else K
        if eps is None:
            self._check(self._lib.hw1f_fused_moments(self._h, rng._h, S1, S2, K, _ptr(P_mkt), _ptr(f_mkt), n_steps_S1,
                                                     C.c_void_p(d_moments_ptr)))
        else:
            self._check(self._lib.hw1f_fused_fd_moments(self._h, rng._h, S1, S2, K, _ptr(P_mkt), _ptr(f_mkt), eps,
                                                        n_steps_S1, C.c_void_p(d_moments_ptr)))

    def fused_finish(self, d_moments_ptr, n_paths_total, P0S2, eps=None, n_steps_S1=0):
        """finalise a (possibly all-reduced) fused moment vector; eps as passed to fused_moments"""
        P, f, se = (np.zeros(self.n_mat, np.float32) for _ in range(3))
        z, v = ZbcResult(), VegaResult()
        self._check(self._lib.hw1f_fused_finish(self._h, C.c_void_p(d_moments_ptr), n_paths_total, P0S2,
                                                0.0 if eps is None else eps, n_steps_S1, _ptr(P), _ptr(f), _ptr(se),
                                                C.byref(z), C.byref(v)))
        return {"P": P, "f": f, "P_se": se, "zbc": z.as_dict(), "vega": v.as_dict()}

    # -- simulate_paths_show (src/1:156-171) --
    def sample_paths(self, rng, n_show=32):
        out = np.zeros((n_show, self.n_steps + 1), np.float32)
        self._check(self._lib.hw1f_sample_paths(self._h, rng._h, n_show, _ptr(out)))
        return out

    # -- benchmark_kernel (src/benchmark_reductions.cu:17-72) --
    def reduction_bench(self, rng, method, P_mkt, f_mkt, S1=5.0, S2=10.0, K=None, n_steps_S1=-1, n_warmup=2,
                        n_runs=5):
        P_mkt, f_mkt = _f32(P_mkt, self.n_mat), _f32(f_mkt, self.n_mat)
        ms, price = C.c_float(), C.c_float()
        self._check(self._lib.hw1f_reduction_bench(self._h, rng._h, method, S1, S2,
                                                   self.K_DEFAULT if K is None else K, _ptr(P_mkt), _ptr(f_mkt),
                                                   n_steps_S1, n_warmup, n_runs, C.byref(ms), C.byref(price)))
        return {"avg_ms": ms.value, "price": price.value}

    def pipe_probe(self, which, iters=256):
        """pipe micro-benchmark: returns (ms, thread-instructions executed)."""
        ms, n = C.c_float(), C.c_double()
        self._check(self._lib.hw1f_pipe_probe(self._h, which, iters, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    # -- parity-test introspection --
    def debug_rng(self, rng, path, n_draws):
        state = np.zeros(6, np.uint32)
        draws = np.zeros(max(n_draws, 1), np.uint32)
        self._check(self._lib.hw1f_debug_rng(self._h, rng._h, int(path), n_draws, _ptr(state), _ptr(draws)))
        return state, draws[:n_draws]

    def debug_normals(self, rng, path, n):
        out = np.zeros(n, np.float32)
        self._check(self._lib.hw1f_debug_normals(self._h, rng._h, int(path), n, _ptr(out)))
        return out
