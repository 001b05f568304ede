"""The double-precision reference (tests/f64_reference.py) against the float oracle (CPU only).

1. Both define the same estimators: their moments agree under cap_oracle.moment_bound on the default model.
2. The pathwise tangent recursion equals a double central difference in sigma on shifted-drift paths.
3. Pair by pair, the oracle's float arithmetic (the engine's reference order) stays inside pair_bound -- the per-pair
   bound derived from operation counts in f64_reference.rel_bound -- on every model the GPU file uses; the bound is the
   per-pair accuracy include/hw1f.h states (a function of |I|, sd(I) and the step count).
4. The drift tables the engine builds (the reference's float expressions) are measured against the exact integrals.
"""
import numpy as np
import pytest

import cap_oracle
import swaption_oracle
import swaption_vega_oracle
from cap_closed_form import continuous_theta
from f64_reference import F64, atm_book, caplet_book, mom5, pair_bound, rel_bound
from oracle_lib import Oracle

SEED = 4242
NP = 1 << 14

# the models of tests/test_gpu_f64.py
SWEEP = [dict(a=a, sigma=s) for a in (1.0, 0.1, 0.05, 0.01, 0.001) for s in (0.01, 0.1)]
MODELS = [dict(), continuous_theta(), dict(n_steps=8184, n_mat=1024, T_final=8.184), dict(n_steps=2, n_mat=3, T_final=0.5)]


def mid(o):
    return 0.5 * o.p.T_final


@pytest.fixture(scope="module")
def dflt():
    o = Oracle()
    P, f = o.bond_curve(SEED, NP)
    return o, F64(o), P, f


def within(got, ref, bound, what):
    gap = np.abs(np.asarray(got) - np.asarray(ref))
    r = float((gap / bound).max())
    print(f"{what}: worst gap / bound {r:.3g}")
    assert (gap <= bound).all(), (what, r)


# ---------------------------------------------------------------- 1. same estimators
def test_curve_moments(dflt):
    o, F, _, _ = dflt
    s, q = o.bond_curve_sums(SEED + 1, NP, first_path=3, offset=1)
    p0, _ = F.curve(SEED + 1, NP, first_path=3, offset=1)
    within(s[1:], p0[:, 1:].sum(0), 3e-6 * s[1:], "curve sum p0")
    within(q[1:], (p0[:, 1:] ** 2).sum(0), 3e-6 * q[1:], "curve sum p0^2")


def zbc_mom(z):
    x, y = z["x"], z["y"]
    return np.array([x.sum(), y.sum(), (x * x).sum(), (y * y).sum(), (x * y).sum()])


def test_zbc_and_vega_fd_moments(dflt):
    o, F, P, f = dflt
    n = o.steps_to(5.0)
    ref = o.zbc_moments(SEED + 2, NP, P, f, offset=1)
    got = zbc_mom(F.zbc(SEED + 2, NP, P, f, n, offset=1))
    within(got, ref, cap_oracle.moment_bound(ref[None])[0], "ZBC")
    eps = 1e-3
    for sc, sg in zip(F.vega_fd(SEED + 2, NP, P, f, n, eps=eps), (o.p.sigma - np.float32(eps), o.p.sigma + np.float32(eps))):
        sg = float(np.float32(sg))
        ref = o.zbc_moments(SEED + 2, NP, P, f, sigma=sg, drift=o.shifted_drift_table(sg))
        within(zbc_mom(sc), ref, cap_oracle.moment_bound(ref[None])[0], f"vega_fd scenario sigma = {sg}")


def test_pathwise_moments(dflt):
    o, F, P, f = dflt
    n = o.steps_to(5.0)
    s, sq = o.vega_pathwise_sums(SEED + 3, NP, P, f, offset=1)
    pw = F.pathwise(SEED + 3, NP, P, f, n, offset=1)
    v = pw["v"][:, 0]
    # rel on the smooth terms, and eps y for a pair whose indicator P > K may flip (moment_bound's argument)
    bound = 3e-6 * np.abs(pw["term1"][:, 0]).sum() + 3e-6 * np.abs(pw["term2"][:, 0]).sum()
    within(s, v.sum(), bound, "pathwise sum v")


def test_cap_and_swaption_moments(dflt):
    o, F, P, f = dflt
    for kind in ("cap", "floor"):
        sw, fl = caplet_book(F, P, [25, 100, 100, 250, 500, 750, 975], 25, kind=kind)
        caps = np.zeros(len(sw), [("T_reset", np.float32), ("T_pay", np.float32), ("K", np.float32),
                                  ("N", np.float32), ("n_steps_reset", np.int32)])
        caps["T_reset"], caps["T_pay"], caps["K"], caps["N"] = sw["T_exercise"], fl["T"], sw["K"], sw["N"]
        caps["n_steps_reset"] = sw["step"]
        ref = cap_oracle.cap_moments(o, SEED + 4, NP, caps, P, f, kind=kind, offset=1)
        bk = F.book(SEED + 4, NP, sw, fl, P, f, offset=1)
        within(mom5(bk["X"], bk["Y"]), ref, cap_oracle.moment_bound(ref), f"{kind} strip")
    sw, fl = atm_book(F, P, [100, 100, 300, 500, 500, 700], [50, 100, 25, 100, 50, 100], [0, 1, 0, 1, 0, 1],
                      big_flows=2048)
    ref = swaption_oracle.swaption_moments(o, SEED + 5, NP // 4, sw, fl, P, f, offset=1)
    bk = F.book(SEED + 5, NP // 4, sw, fl, P, f, offset=1)
    within(mom5(bk["X"], bk["Y"]), ref, cap_oracle.moment_bound(ref), "swaption book")
    eps = 1e-3
    mom, aux = swaption_vega_oracle.vega_moments(o, SEED + 6, NP // 4, sw, fl, P, f, eps, offset=1)
    _, vref = swaption_vega_oracle.split(mom, len(sw))
    bv = F.book_vega(SEED + 6, NP // 4, sw, fl, P, f, eps, offset=1)
    got = np.stack([bv["Xm"].sum(0), (bv["Xm"] ** 2).sum(0), bv["Xp"].sum(0), (bv["Xp"] ** 2).sum(0),
                    bv["D"].sum(0), (bv["D"] ** 2).sum(0)], axis=1)
    bound = swaption_vega_oracle.vega_bound(vref, aux)
    within(got[:, [0, 2, 4]], vref[:, [0, 2, 4]], bound[:, [0, 2, 4]], "book vega X-, X+, D")


# ---------------------------------------------------------------- 2. tangent vs central difference
@pytest.mark.parametrize("over", [dict(), dict(a=0.1), dict(a=0.01, sigma=0.01)], ids=str)
def test_tangent_equals_central_difference(over):
    o = Oracle(**over)
    F = F64(o)
    P, f = o.bond_curve(SEED, 1 << 10)
    n, h = o.steps_to(5.0), F.sigma * 1e-5
    pw = F.pathwise(SEED + 7, 512, P, f, n)
    cd = F.pathwise_cd(SEED + 7, 512, P, f, n, h=h)
    # pairs whose payoff crosses the kink inside the bump are not differentiable there
    z = pw["zbc"]
    far = np.abs(z["P"] - Oracle.K_DEFAULT) > 4 * h * np.abs(z["P"] * z["B"] * (np.abs(pw["t"]) + F.sigma * z["B"]))
    assert far.mean() > 0.9
    gap = np.abs(pw["v"] - cd)[far]
    scale = np.abs(pw["term1"]).max() + np.abs(pw["term2"]).max()
    print(f"{over}: tangent vs central difference, worst gap {gap.max():.3g} (scale {scale:.3g})")
    assert gap.max() <= 1e-8 * max(scale, 1e-3)


# ---------------------------------------------------------------- 3. float arithmetic per pair
def oracle_pairs(o, F, P, f, n_pairs, first_path, offset, drift):
    """per pair: the float oracle's curve and ZBC summands and the f64 ones, with their bounds"""
    n = max(1, min(o.steps_to(mid(o)), o.p.n_steps))
    S1 = float(np.float32(n * np.float32(o.dt)))
    cur, zx, zy = [], [], []
    st = F.states(SEED + 8, n_pairs, np.arange(1, F.n_mat) * F.stride, first_path, offset, drift=drift)
    p0 = np.exp(-st[:, :, 2]) + np.exp(-st[:, :, 3])
    T = np.arange(1, F.n_mat) * F.stride * F.dt
    z = F.zbc(SEED + 8, n_pairs, P, f, n, S1=S1, S2=o.p.T_final, first_path=first_path, offset=offset, drift=drift)
    for q in range(n_pairs):
        s, _ = o.bond_curve_sums(SEED + 8, 1, first_path=first_path + q, offset=offset)
        cur.append(s[1:])
        m = o.zbc_moments(SEED + 8, 1, P, f, S1=S1, S2=o.p.T_final, n_steps_S1=n, first_path=first_path + q,
                          offset=offset)
        zx.append(m[0])
        zy.append(m[1])
    Iabs = np.maximum(np.abs(st[:, :, 2]), np.abs(st[:, :, 3]))
    rel_c = rel_bound(np.arange(1, F.n_mat) * F.stride, Iabs, np.array([F.sd_I(t) for t in T]))
    rel_z = rel_bound(n, z["I_abs"].max(1), F.sd_I(S1), r_abs=z["r_abs"].max(1), B=z["B"], sd_r=F.sd_r(S1))
    X, Y = z["x"].sum(1), z["y"].sum(1)
    return (np.array(cur), p0, pair_bound(p0, rel_c), rel_c, np.array(zx), X, pair_bound(X, rel_z, Y),
            np.array(zy), Y, pair_bound(Y, rel_z), rel_z)


def pair_report(o, F, P, f, drift, what):
    cur, p0, cb, rc, zx, X, xb, zy, Y, yb, rz = oracle_pairs(o, F, P, f, 48, 1000, 1, drift)
    worst = {"curve": float((np.abs(cur - p0) / cb).max()), "zbc X": float((np.abs(zx - X) / xb).max()),
             "zbc Y": float((np.abs(zy - Y) / yb).max())}
    rel_err = np.abs(cur / p0 - 1)
    print(f"{what}: per-pair |oracle / f64 - 1| of p0: median {np.median(rel_err):.2e}, 99% {np.quantile(rel_err, .99):.2e}, "
          f"max {rel_err.max():.2e}; worst gap / pair_bound {worst}; rel bound max {max(rc.max(), rz.max()):.2e}")
    return worst, max(rc.max(), rz.max())


@pytest.mark.parametrize("over", MODELS, ids=lambda o: "-".join(f"{k}{v}" for k, v in o.items()) or "default")
def test_oracle_pairs_within_bound(over):
    o = Oracle(**over)
    F = F64(o)
    P, f = o.bond_curve(SEED, 1 << 10)
    worst, rel = pair_report(o, F, P, f, None, str(over))
    assert max(worst.values()) <= 0.5      # the oracle uses well under the bound
    if o.p.n_steps == 1000:
        # the bound is a function of the pair's |I|, sd(I) and the step count (include/hw1f.h states it); on 1000 steps
        # of the default parameters it is at most 1.3e-5, for the pair with the largest |I|
        assert rel <= 1.3e-5


@pytest.mark.parametrize("over", SWEEP, ids=lambda o: f"a{o['a']}-s{o['sigma']}")
def test_oracle_pairs_sweep(over):
    """The a / sigma sweep on 1000 x 101: the path arithmetic, on the engine's own drift table, within the bound.  The
    drift table is measured separately (test_float_drift_table_error)."""
    o = Oracle(**over)
    F = F64(o)
    P, f = o.bond_curve(SEED, 1 << 10)
    d, _ = o.drift_tables()
    worst, rel = pair_report(o, F, P, f, d.astype(np.float64), f"{over} (engine drift table)")
    # the bound grows with |I| (float rounding is relative to |I|): printed above, 3.5e-6 to 4.7e-5 over the sweep
    assert max(worst.values()) <= 1.0


# ---------------------------------------------------------------- 4. the float drift tables
# |I_table - I_exact| of the noise-free path at T_final = 10 (dt = 0.01), where the engine's drift table (the
# reference's compute_drift_tables in float: (1 - e^{-a dt}) / a and ((s + dt) - e s) / a - (1 - e) / a^2 lose
# their digits as a dt -> 0) replaces the exact integrals: measured 3.4e-8, 5.5e-6, 1.2e-5, 1.1e-3, 8.7e-2.
# Upper bounds only: a table computed more accurately passes.
TABLE_ERR = {1.0: 2e-6, 0.1: 1e-5, 0.05: 5e-5, 0.01: 2e-3, 0.001: 0.15}


@pytest.mark.parametrize("a", sorted(TABLE_ERR), ids=lambda a: f"a{a}")
def test_float_drift_table_error(a):
    o = Oracle(a=a)
    F = F64(o)
    d, _ = o.drift_tables()

    def I(tab):
        m, acc = F.r0, 0.0
        for x in tab:
            mn = m * F.e + float(x)
            acc += 0.5 * (m + mn) * F.dt
            m = mn
        return acc
    err = abs(I(d.astype(np.float64)) - I(F.drift()))
    print(f"a = {a}: noise-free |I(10)| table vs exact {err:.3g}")
    assert err <= TABLE_ERR[a]
    if a >= 0.1:       # below, the table, not the path arithmetic, limits the accuracy (include/hw1f.h)
        assert err <= 1e-5
