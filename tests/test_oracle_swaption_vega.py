"""Vega of a swaption book on the CPU: the book vega oracle (tests/swaption_vega_oracle.c, three sigma scenarios on the
same normals in reference order) against the swaption book oracle and against Jamshidian's closed form differenced at
sigma -/+ eps on the same curve."""
import numpy as np
import pytest

import swaption_oracle
import swaption_vega_oracle as svo
from cap_closed_form import continuous_theta
from swaption_closed_form import book_closed_form, par_rate

N_CURVE = 1 << 16
N_SW = 1 << 13
EPS = 1e-3


def test_base_block_is_the_swaption_oracle(hw):
    """default params (theta_a1 != fd_theta_a1), exercises before and after theta_break; one OpenMP thread, so that both
    oracles sum their pairs in the same order"""
    from oracle_lib import Oracle
    o = Oracle()
    s, _ = o.bond_curve_sums(5, 1 << 12)
    P, f = o.curve_finalize(s, 1 << 12)
    sw, fl = hw.swaption_schedule([1.0, 4.0, 6.0, 6.0], [3.0, 5.0, 2.0, 4.0], 0.05, freq=2, notional=100.0,
                                  kind=["payer", "receiver", "payer", "receiver"])
    threads = o.max_threads()
    svo.set_threads(1)
    try:
        mom, _ = svo.vega_moments(o, 77, 1 << 10, sw, fl, P, f, EPS, offset=3)
        ref = swaption_oracle.swaption_moments(o, 77, 1 << 10, sw, fl, P, f, offset=3)
    finally:
        svo.set_threads(threads)
    base, vega = svo.split(mom, len(sw))
    assert np.array_equal(base, ref)
    assert (vega[:, [1, 3, 5]] > 0).all()
    # the book's first moments are the sums over its options
    assert vega[-1, 0] == pytest.approx(vega[:-1, 0].sum(), rel=1e-12)
    assert vega[-1, 4] == pytest.approx(vega[:-1, 4].sum(), rel=1e-12)


@pytest.fixture(scope="module")
def model():
    from oracle_lib import Oracle
    o = Oracle(**continuous_theta())
    s, q = o.bond_curve_sums(778, N_CURVE)
    P, f = o.curve_finalize(s, N_CURVE)
    n = float(N_CURVE)
    x, xx = 0.5 * s, 0.25 * q
    P_se = np.sqrt(np.maximum((xx - x * x / n) / (n - 1), 0.0) / n).astype(np.float32)
    P_se[0] = 0.0
    return o, P, f, P_se


def test_oracle_vega_vs_jamshidian(hw, model):
    o, P, f, P_se = model
    Tf, a, sigma = float(o.p.T_final), float(o.p.a), float(o.p.sigma)
    Te = np.array([1.0, 1.0, 2.0, 3.0, 5.0, 5.0, 7.0])
    ten = np.array([2.0, 5.0, 3.0, 4.0, 5.0, 2.0, 3.0])
    kappa = [par_rate(P, Tf, t, n, 2) + d for t, n, d in zip(Te, ten, (0.0, 0.01, -0.01, 0.0, 0.005, 0.0, -0.005))]
    kinds = ["payer", "receiver", "payer", "receiver", "payer", "payer", "receiver"]
    sw, fl = hw.swaption_schedule(Te, ten, kappa, freq=2, notional=100.0, kind=kinds)
    mom, _ = svo.vega_moments(o, 4243, N_SW, sw, fl, P, f, EPS)
    _, vb = svo.split(mom, len(sw))
    eps32 = float(np.float32(EPS))
    sm, sp = float(np.float32(sigma - eps32)), float(np.float32(sigma + eps32))

    def cf(P_, s_):
        return np.array(book_closed_form(sw, fl, P_, f, a, s_, Tf))

    def vega_cf(P_):
        return (cf(P_, sp) - cf(P_, sm)) / (2 * eps32)
    want, want_m, want_p = vega_cf(P), cf(P, sm), cf(P, sp)
    allow = np.abs(vega_cf(P + P_se) - vega_cf(P - P_se))
    allow_m, allow_p = np.abs(cf(P + P_se, sm) - cf(P - P_se, sm)), np.abs(cf(P + P_se, sp) - cf(P - P_se, sp))
    worst = 0.0
    for i in range(len(sw)):
        r = svo.vega_algebra(vb[i], N_SW, eps32)
        worst = max(worst, abs(r["vega"] - want[i]) / (4 * r["vega_se"] + allow[i]))
        assert abs(r["vega"] - want[i]) <= 4 * r["vega_se"] + allow[i], (i, r, want[i], allow[i])
        assert abs(r["price_minus"] - want_m[i]) <= 4 * r["se_minus"] + allow_m[i], (i, r, want_m[i])
        assert abs(r["price_plus"] - want_p[i]) <= 4 * r["se_plus"] + allow_p[i], (i, r, want_p[i])
        assert r["vega"] > 0 and r["vega_se"] < 0.2 * r["vega"], (i, r)
    r = svo.vega_algebra(vb[-1], N_SW, eps32)
    assert abs(r["vega"] - want.sum()) <= 4 * r["vega_se"] + allow.sum(), (r, want.sum())
    print(f"worst |vega - Jamshidian| / (4 se + allowance) {worst:.3g}")
