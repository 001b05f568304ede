"""Double-precision reference of the engine's discrete scheme, pair by pair (tests/f64_reference.c walks the paths).

TEST INFRASTRUCTURE.  The float oracle (oracle/hw1f_oracle.c) re-executes the engine's float recipe; this module
evaluates the same estimators in double from the model's parameters, so that an error the oracle and a kernel share --
a drift convention, a factor of the bond variance, a cancellation in float -- shows up, and so that single pairs of
paths can be compared.  The shared library is compiled on first use into the temporary directory, keyed by a hash of
its sources, like the other oracles.

What is computed in double here: the Box-Muller normals (log, sqrt, sin, cos), the drift tables (the integrals of the
piecewise-linear theta restated, not the float expressions), the recursion of r and of the trapezoid integral I, the
bond plans P(t, T) = P_M(T) / P_M(t) exp(B f_M(t) - sigma^2 / (4 a) (1 - e^{-2 a t}) B^2 - B r), payoffs and controls.

Shared conventions (deliberately the engine's, so that both sides compute the same estimator):
  - P_M and f_M are interpolated linearly between the knots k T_final / (n_mat - 1) of the float curves passed in and
    clamped at the last knot;
  - dt, e^{-a dt} (the step decay) and sig_st (the step standard deviation of each sigma scenario) are the float values
    the engine uses; the model's float parameters are read as the doubles they are;
  - the theta piece of step i is the one of its left end, chosen as the engine chooses it (float i dt < theta_break);
  - the finite-difference ZBC scenarios of hw1f_vega_fd keep fd_theta_a1 for t >= theta_break, because the engine
    defines them that way; the book vega's bumped scenarios use theta_a1.

Every estimator returns per-pair summands (the quantities whose sums the kernels return), not only moments.
"""
import ctypes as C
import hashlib
import math
import os
import subprocess
import tempfile

import numpy as np

from cap_oracle import CFLAGS, ORACLE_DIR
from oracle_lib import Oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "f64_reference.c"), os.path.join(ORACLE_DIR, "xorwow_ref.c"),
           os.path.join(ORACLE_DIR, "xorwow_ref.h")]

U = 2.0 ** -24          # unit roundoff of float
EPS_EX2 = 2.4e-7        # MUFU.EX2 vs exp (2 ulp): cap_oracle.moment_bound's eps
# Allowance for the error of one normal G = s sin v (MUFU.LG2 / SQRT / SIN / COS on the GPU, libm in float on the CPU).
# From the PTX specification: sin/cos.approx err by at most 2^-20.5 absolute, lg2.approx and sqrt.approx by about 2^-22
# relative, so |dG| <= 2^-20.5 s + 2^-22 |G|, 1.2e-6 at the rms radius s = sqrt 2.  The bound sums these errors as if
# they were independent, and they are not: the MUFU error is a smooth function of the angle.  At 1.2e-6 two B200 pairs
# in tests/test_gpu_f64.py came out at 1.2x and 1.3x the bound (pathwise on 8184 x 1024 at path 2^32 + 530, and ZBC at
# a = 0.001, sigma = 0.1 in reference order, both in the file), so the allowance is widened to 2e-6.
DELTA_G = 2e-6
K_SIGMA = 5.0           # per-pair bounds are 5-sigma bounds of sums of independent roundings

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as fh:
            h.update(fh.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), f"hw1f_f64_reference_{os.getuid()}")
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, f"libhw1f_f64_reference_{h.hexdigest()[:16]}.so")
    if not os.path.exists(path):
        tmp = f"{path}.{os.getpid()}.tmp"
        subprocess.check_call(["gcc"] + CFLAGS + ["-shared", "-I", ORACLE_DIR, "-o", tmp, SOURCES[0], SOURCES[1], "-lm"],
                              stdout=subprocess.DEVNULL)
        os.replace(tmp, path)   # atomic: concurrent test processes see a complete library or none
    return path


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.f64_normals.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int, C.c_void_p]
        _lib.f64_pair_states.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, C.c_uint64,
                                         C.c_uint64, C.c_int64, C.c_uint64, C.c_void_p, C.c_int, C.c_void_p]
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _E(x):
    """1 - e^{-x} without cancellation"""
    return -np.expm1(-np.asarray(x, np.float64))


class F64:
    """The model of an Oracle (same float parameters) evaluated in double."""

    def __init__(self, oracle: Oracle):
        self.o = oracle
        p = oracle.p
        self.a, self.sigma, self.r0, self.T_final = float(p.a), float(p.sigma), float(p.r0), float(p.T_final)
        self.n_steps, self.n_mat = int(p.n_steps), int(p.n_mat)
        self.stride = self.n_steps // (self.n_mat - 1)
        self.dt = float(oracle.dt)
        self.e = float(oracle.L.orc_exp_adt(C.byref(p)))
        self.spacing = self.T_final / (self.n_mat - 1)
        i = np.arange(self.n_steps)
        self.s = i * self.dt
        self.t = (i + 1) * self.dt
        self.piece1 = (i.astype(np.float32) * np.float32(self.dt)) >= np.float32(p.theta_break)

    # ---- model tables -----------------------------------------------------------------
    def sig_st(self, sigma=None):
        return float(self.o.sig_st(self.sigma if sigma is None else sigma))

    def drift(self, sigma_new=None, a1=None):
        """int_s^t e^{-a (t - u)} theta(u) du per step (theta = a0 + b0 u, or a1 + b1 u on the second piece), plus, for
        sigma_new, the shift of run_finite_difference: (sigma_new^2 - sigma^2) / (2 a^2) (1 - e^{-a dt})(1 - e^{-a(t+s)})"""
        p, a, s = self.o.p, self.a, self.s
        A = np.where(self.piece1, float(p.theta_a1 if a1 is None else a1), float(p.theta_a0))
        Bt = np.where(self.piece1, float(p.theta_b1), float(p.theta_b0))
        E = _E(a * self.dt)
        # int_s^t e^{-a(t-u)} du = E / a;  int_s^t e^{-a(t-u)} u du = s E / a + (dt - E / a) / a
        d = A * E / a + Bt * (s * E / a + (self.dt - E / a) / a)
        if sigma_new is not None:
            d = d + (float(sigma_new) ** 2 - self.sigma ** 2) / (2 * a * a) * E * _E(a * (self.t + s))
        return d

    def sdrift(self, sigma=None):
        """d/dsigma of the shifted drift at sigma_new = sigma: the tangent's drift"""
        sigma = self.sigma if sigma is None else float(sigma)
        return sigma / (self.a * self.a) * _E(self.a * self.dt) * _E(self.a * (self.t + self.s))

    def interp(self, data, T):
        data = np.asarray(data, np.float64)
        x = float(T) / self.spacing
        k = int(math.floor(x))
        if k >= self.n_mat - 1:
            return float(data[-1])
        w = x - k
        return float((1 - w) * data[k] + w * data[k + 1])

    def bond_plan(self, sigma, t, T, P_mkt, f_mkt):
        """(A, B) of P(t, T) = A e^{-B r}"""
        a = self.a
        B = float(_E(a * (T - t))) / a
        var = sigma * sigma / (4 * a) * float(_E(2 * a * t)) * B * B
        A = self.interp(P_mkt, T) / self.interp(P_mkt, t) * math.exp(B * self.interp(f_mkt, t) - var)
        return A, B

    # ---- paths ---------------------------------------------------------------------------
    def states(self, seed, n_pairs, eval_steps, first_path=0, offset=0, drift=None, sig_st=None, r0=None):
        """[n_pairs, len(eval_steps), 4]: r(+G), r(-G), I(+G), I(-G) after each eval step"""
        drift = np.ascontiguousarray(self.drift() if drift is None else drift, np.float64)
        steps = np.ascontiguousarray(eval_steps, np.int32)
        assert len(steps) and (np.diff(steps) >= 0).all() and steps[-1] <= len(drift)
        out = np.zeros((n_pairs, len(steps), 4), np.float64)
        lib().f64_pair_states(_p(drift), self.e, self.dt, self.sig_st() if sig_st is None else sig_st,
                              self.r0 if r0 is None else r0, seed, first_path, n_pairs, offset, _p(steps), len(steps),
                              _p(out))
        return out

    def normals(self, seed, subsequence, offset, n):
        out = np.zeros(n, np.float64)
        lib().f64_normals(seed, subsequence, offset, n, _p(out))
        return out

    def sd_I(self, T, sigma=None):
        """standard deviation of the noise part of I(T) (continuous time): sizes the normals' error allowance"""
        a, sigma = self.a, self.sigma if sigma is None else sigma
        v = T - 2 * float(_E(a * T)) / a + float(_E(2 * a * T)) / (2 * a)
        return sigma / a * math.sqrt(max(v, 0.0))

    def sd_r(self, T, sigma=None):
        a, sigma = self.a, self.sigma if sigma is None else sigma
        return sigma * math.sqrt(float(_E(2 * a * T)) / (2 * a))

    # ---- estimators: per-pair summands -----------------------------------------------------
    def curve(self, seed, n_pairs, first_path=0, offset=0):
        """p0[n_pairs, n_mat] = e^{-I(+G)} + e^{-I(-G)} at every save point (column 0: 2); I_abs: max |I| per entry"""
        steps = np.arange(1, self.n_mat) * self.stride
        st = self.states(seed, n_pairs, steps, first_path, offset)
        p0 = np.full((n_pairs, self.n_mat), 2.0)
        p0[:, 1:] = np.exp(-st[:, :, 2]) + np.exp(-st[:, :, 3])
        I_abs = np.zeros((n_pairs, self.n_mat))
        I_abs[:, 1:] = np.maximum(np.abs(st[:, :, 2]), np.abs(st[:, :, 3]))
        return p0, I_abs

    def zbc(self, seed, n_pairs, P_mkt, f_mkt, n_steps_S1, S1=5.0, S2=10.0, K=None, first_path=0, offset=0,
            sigma=None, drift=None):
        """per twin x = D (P - K)^+, y = D P at step n_steps_S1: dict of [n_pairs, 2] arrays (+G, -G) and I_abs"""
        sigma = self.sigma if sigma is None else float(sigma)
        K = Oracle.K_DEFAULT if K is None else K
        st = self.states(seed, n_pairs, [n_steps_S1], first_path, offset, drift=drift, sig_st=self.sig_st(sigma))[:, 0]
        A, B = self.bond_plan(sigma, S1, S2, P_mkt, f_mkt)
        P = A * np.exp(-B * st[:, :2])
        D = np.exp(-st[:, 2:])
        return {"x": D * np.maximum(P - K, 0.0), "y": D * P, "P": P, "D": D, "B": B,
                "I_abs": np.abs(st[:, 2:]), "r_abs": np.abs(st[:, :2])}

    def pathwise(self, seed, n_pairs, P_mkt, f_mkt, n_steps_S1, S1=5.0, S2=10.0, K=None, first_path=0, offset=0):
        """per twin v = d/dsigma [D (P - K)^+] by the tangent recursion: [n_pairs, 2], plus the parts of the bound"""
        K = Oracle.K_DEFAULT if K is None else K
        z = self.zbc(seed, n_pairs, P_mkt, f_mkt, n_steps_S1, S1, S2, K, first_path, offset)
        tg = self.states(seed, n_pairs, [n_steps_S1], first_path, offset, drift=self.sdrift(),
                         sig_st=self.sig_st() / self.sigma, r0=0.0)[:, 0]
        t, J = tg[:, :2], tg[:, 2:]
        a, B = self.a, z["B"]
        xk = self.sigma / (2 * a) * float(_E(2 * a * S1))
        dP = -z["P"] * B * (xk * B + t)
        term1 = np.where(z["P"] > K, z["D"] * dP, 0.0)
        term2 = z["x"] * J
        return {"v": term1 - term2, "term1": term1, "term2": term2, "zbc": z, "t": t, "J": J}

    def pathwise_cd(self, seed, n_pairs, P_mkt, f_mkt, n_steps_S1, S1=5.0, S2=10.0, K=None, first_path=0, offset=0,
                    h=None):
        """the same derivative as a central difference in sigma on shifted-drift paths (theta_a1 kept): [n_pairs, 2]"""
        h = self.sigma * 1e-5 if h is None else h
        x = []
        for sg in (self.sigma - h, self.sigma + h):
            st = self.states(seed, n_pairs, [n_steps_S1], first_path, offset, drift=self.drift(sigma_new=sg),
                             sig_st=self.sig_st() * sg / self.sigma)[:, 0]
            A, B = self.bond_plan(sg, S1, S2, P_mkt, f_mkt)
            x.append(np.exp(-st[:, 2:]) * np.maximum(A * np.exp(-B * st[:, :2]) - (Oracle.K_DEFAULT if K is None else K),
                                                     0.0))
        return (x[1] - x[0]) / (2 * h)

    def vega_fd(self, seed, n_pairs, P_mkt, f_mkt, n_steps_S1, eps=1e-3, **kw):
        """hw1f_vega_fd's scenarios: ZBC at sigma -/+ eps on the shifted drift with fd_theta_a1 (the engine's quirk)"""
        a1 = float(self.o.p.fd_theta_a1)
        return [self.zbc(seed, n_pairs, P_mkt, f_mkt, n_steps_S1, sigma=sg,
                         drift=self.drift(sigma_new=sg, a1=a1), **kw) for sg in
                (float(np.float32(self.sigma - np.float32(eps))), float(np.float32(self.sigma + np.float32(eps))))]

    def book(self, seed, n_pairs, sw, flows, P_mkt, f_mkt, first_path=0, offset=0, sigma=None, drift=None):
        """a book of coupon-bond options (swaption_oracle's layout; sw["step"] given): X, Y [n_pairs, n + 1] with
        X = N (x(+G) + x(-G)), Y = N (y(+G) + y(-G)), the book last; Yabs (the kink scale) and the bound's parts"""
        sigma = self.sigma if sigma is None else float(sigma)
        n = len(sw)
        steps = np.asarray(sw["step"], np.int32)
        st = self.states(seed, n_pairs, steps, first_path, offset, drift=drift, sig_st=self.sig_st(sigma))
        X = np.zeros((n_pairs, n + 1))
        Y = np.zeros((n_pairs, n + 1))
        I_abs = np.zeros((n_pairs, n + 1))
        for i in range(n):
            Te = float(sw["T_exercise"][i])
            bnd = np.zeros((n_pairs, 2))
            for j in range(int(sw["first_flow"][i]), int(sw["first_flow"][i]) + int(sw["n_flows"][i])):
                A, B = self.bond_plan(sigma, Te, float(flows["T"][j]), P_mkt, f_mkt)
                bnd += float(flows["c"][j]) * A * np.exp(-B * st[:, i, :2])
            D = np.exp(-st[:, i, 2:])
            sgn = -1.0 if int(sw["kind"][i]) == 0 else 1.0
            N = float(sw["N"][i])
            X[:, i] = N * (D * np.maximum(sgn * (bnd - float(sw["K"][i])), 0.0)).sum(axis=1)
            Y[:, i] = N * (D * bnd).sum(axis=1)
            I_abs[:, i] = np.abs(st[:, i, 2:]).max(axis=1)
        X[:, n], Y[:, n] = X[:, :n].sum(axis=1), Y[:, :n].sum(axis=1)
        I_abs[:, n] = I_abs[:, :n].max(axis=1)
        return {"X": X, "Y": Y, "I_abs": I_abs, "steps": steps}

    def book_vega(self, seed, n_pairs, sw, flows, P_mkt, f_mkt, eps, **kw):
        """X- and X+ of the book at sigma -/+ eps (shifted drift with theta_a1, the curve kept) and D = X+ - X-"""
        out = []
        for sg in (float(np.float32(self.sigma - np.float32(eps))), float(np.float32(self.sigma + np.float32(eps)))):
            out.append(self.book(seed, n_pairs, sw, flows, P_mkt, f_mkt, sigma=sg, drift=self.drift(sigma_new=sg), **kw))
        m, p = out
        return {"Xm": m["X"], "Xp": p["X"], "D": p["X"] - m["X"], "minus": m, "plus": p}


# ---- bounds ----------------------------------------------------------------------------------
def rel_bound(n_steps, I_abs, sd_I, r_abs=0.0, B=0.0, sd_r=0.0, n_flows=1):
    """Relative error a float evaluation of D = e^{-I} times a bond function may carry against the double one, from
    operation counts (6-sigma bounds of sums of independent roundings, each at most u = 2^-24 relative):
      - I accumulates n_steps trapezoid terms, one rounding of |I| each, and every step's shock carries one rounding of
        the normal (DELTA_G, the MUFU or libm allowance) that reaches I through its noise part: u sqrt(n) |I| + DELTA_G sd_I;
      - r carries the same normal errors (DELTA_G sd_r) and one rounding of |r| per step, reaching P through B;
      - a coupon bond sums n_flows terms (one rounding each);
      - e^{-I} and each P = A ex2(..) carry one MUFU.EX2 (EPS_EX2) and the handful of products around them (4 u)."""
    dI = K_SIGMA * (U * np.sqrt(n_steps) * I_abs + DELTA_G * sd_I)
    dr = K_SIGMA * (U * np.asarray(r_abs) + DELTA_G * sd_r) * B
    return dI + dr + K_SIGMA * U * np.sqrt(n_flows) + 2 * EPS_EX2 + 4 * U


def pair_bound(x, rel, y=0.0):
    """Largest |float - f64| of one summand x: rel |x|, plus, for an option payoff, the absolute form at the kink --
    x = D (s (Bnd - K))^+ inherits the ABSOLUTE error of D Bnd, so rel y with y = D Bnd (cap_oracle.moment_bound's
    argument).  A CRN difference X+ - X- gets the sum of its two terms' bounds (pass |X+| + |X-| and y+ + y-)."""
    return rel * (np.abs(x) + np.abs(y))


def mom5(X, Y):
    """the engine's five pair moments of each column: [n + 1, 5]"""
    return np.stack([X.sum(0), Y.sum(0), (X * X).sum(0), (Y * Y).sum(0), (X * Y).sum(0)], axis=1)


# ---- books shared by the CPU and GPU files ------------------------------------------------------
BOOK_DTYPE = np.dtype([("T_exercise", np.float32), ("K", np.float32), ("N", np.float32), ("kind", np.int32),
                       ("n_steps_exercise", np.int32), ("first_flow", np.int32), ("n_flows", np.int32),
                       ("reserved", np.int32), ("step", np.int32)])
FLOWS_DTYPE = np.dtype([("T", np.float32), ("c", np.float32)])


def atm_book(F: F64, P_mkt, exercise_steps, tenor_steps, kinds, big_flows=0):
    """near-the-money coupon-bond options on the step grid: option i exercises at exercise_steps[i] (repeats = gaps of
    0), pays a coupon every tenor_steps[i] steps to T_final (at least one flow), strike 1 and the par coupon of the
    market curve; kinds[i] 0 payer, 1 receiver.  big_flows > 0 appends a receiver whose 'big_flows' flows are spread
    evenly over (T_e, T_final] from the last exercise step."""
    dt, T_final = F.dt, F.T_final
    rows, flows = [], []
    spec = list(zip(exercise_steps, tenor_steps, kinds))
    if big_flows:
        spec.append((exercise_steps[-1], None, 1))
        # the book's flows may not exceed HW1F_MAX_SWAPTION_FLOWS = big_flows in all
        big_flows -= sum(max(1, len(range(k + t, F.n_steps + 1, t))) for k, t, _ in spec[:-1])
    for k, tenor, kind in spec:
        Te = float(np.float32(k * np.float32(dt)))
        if tenor is None:
            T = Te + (T_final - Te) * np.arange(1, big_flows + 1) / big_flows
        else:
            T = np.arange(k + tenor, F.n_steps + 1, tenor) * dt
            if len(T) == 0:
                T = np.array([T_final])
        T = np.unique(np.minimum(np.asarray(T, np.float32), np.float32(T_final)))
        T = T[T > np.float32(Te)]
        taus = np.diff(np.concatenate([[Te], T.astype(np.float64)]))
        Ps = np.array([F.interp(P_mkt, t) for t in T])
        kappa = max((F.interp(P_mkt, Te) - Ps[-1]) / float((taus * Ps).sum()), 1e-3)   # coupons must be positive
        c = (kappa * taus).astype(np.float64)
        c[-1] += 1.0
        rows.append((Te, 1.0, 1.0, kind, k, len(flows), len(T), 0, k))
        flows.extend(zip(T.tolist(), c.tolist()))
    return np.array(rows, BOOK_DTYPE), np.array(flows, FLOWS_DTYPE)


def caplet_book(F: F64, P_mkt, reset_steps, tau_steps, kind="cap"):
    """a strip of near-the-money caplets (kind "cap": bond puts, payer; "floor": bond calls, receiver) as one-flow
    options: reset at reset_steps[i], paid tau_steps later (capped at T_final), bond strike K = P_M(T_p) / P_M(T_r)"""
    rows, flows = [], []
    for i, k in enumerate(reset_steps):
        Tr = float(np.float32(k * np.float32(F.dt)))
        Tp = float(np.float32(min((k + tau_steps) * F.dt, F.T_final)))
        K = F.interp(P_mkt, Tp) / F.interp(P_mkt, Tr)
        rows.append((Tr, K, 1.0, 0 if kind == "cap" else 1, k, i, 1, 0, k))
        flows.append((Tp, 1.0))
    return np.array(rows, BOOK_DTYPE), np.array(flows, FLOWS_DTYPE)


def book_rel(F: F64, bk, sw, n_steps_col=None):
    """rel_bound of each column of F.book's output (the options, then the book), per pair"""
    n = len(sw)
    rel = np.zeros_like(bk["X"])
    for i in range(n + 1):
        j = min(i, n - 1) if i < n else int(np.argmax(sw["step"]))
        k = int(sw["step"][j]) if i < n else int(sw["step"].max())
        nf = int(sw["n_flows"][j]) if i < n else int(sw["n_flows"].max())
        rel[:, i] = rel_bound(k, bk["I_abs"][:, i], F.sd_I(k * F.dt), r_abs=0.1, B=F.T_final, sd_r=F.sd_r(k * F.dt),
                              n_flows=nf)
    return rel
