"""European swaptions on the CPU: the book oracle (tests/swaption_oracle.c, the reference-order float sequence evaluated
at every exercise step) against Jamshidian's closed form, the closed form's own identities, and swaption_schedule."""
import math

import numpy as np
import pytest

import swaption_oracle
from cap_closed_form import bond_option, continuous_theta, interp_mkt, pair_algebra
from swaption_closed_form import (book_closed_form, flows_of, forward_swap, hw_bond_coeffs, jamshidian_rstar, par_rate,
                                  swaption_price)

N_CURVE = 1 << 16
N_SW = 1 << 13


def test_swaption_schedule_flows(hw):
    sw, fl = hw.swaption_schedule([1.0, 2.0, 2.0], [2.0, 1.0, 1.5], 0.03, freq=2, notional=[100.0, 200.0, 300.0],
                                  kind=["payer", "receiver", "payer"])
    assert sw.dtype.itemsize == 32 and fl.dtype.itemsize == 8
    assert list(sw["kind"]) == [hw._ffi.KIND_PAYER, hw._ffi.KIND_RECEIVER, hw._ffi.KIND_PAYER]
    assert (sw["K"] == 1.0).all() and (sw["n_steps_exercise"] == -1).all()
    np.testing.assert_array_equal(sw["N"], [100.0, 200.0, 300.0])
    np.testing.assert_array_equal(sw["first_flow"], [0, 4, 6])
    np.testing.assert_array_equal(sw["n_flows"], [4, 2, 3])
    np.testing.assert_array_equal(fl["T"], np.float32([1.5, 2.0, 2.5, 3.0, 2.5, 3.0, 2.5, 3.0, 3.5]))
    want_c = np.float32([0.015, 0.015, 0.015, 1.015, 0.015, 1.015, 0.015, 0.015, 1.015])
    np.testing.assert_array_equal(fl["c"], want_c)
    # annual, one kind for all, a scalar expiry broadcast over tenors
    sw, fl = hw.swaption_schedule(3.0, [1, 2], 0.05, kind="receiver")
    assert (sw["kind"] == hw._ffi.KIND_RECEIVER).all() and list(sw["n_flows"]) == [1, 2]
    np.testing.assert_array_equal(fl["T"], np.float32([4.0, 4.0, 5.0]))
    np.testing.assert_array_equal(fl["c"], np.float32([1.05, 0.05, 1.05]))
    with pytest.raises(ValueError):
        hw.swaption_schedule(1.0, 0.3, 0.02, freq=2)     # not a whole number of coupon periods


def test_jamshidian_one_flow_is_the_bond_option(hw):
    from oracle_lib import Oracle
    o = Oracle(**continuous_theta())
    s, _ = o.bond_curve_sums(5, 1 << 12)
    P, f = o.curve_finalize(s, 1 << 12)
    a, sigma, Tf = float(o.p.a), float(o.p.sigma), float(o.p.T_final)
    n = len(P)
    for Te, T, K in ((1.0, 2.0, 0.97), (3.0, 8.0, 0.8), (5.0, 10.0, 0.9)):
        for kind, bk in (("payer", "cap"), ("receiver", "floor")):
            want = bond_option(bk, interp_mkt(P, Te, Tf, n), interp_mkt(P, T, Tf, n), K, a, sigma, Te, T)
            got = swaption_price(kind, P, f, a, sigma, Tf, Te, [T], [1.0], K, N=1.0)
            assert got == pytest.approx(want, rel=1e-12, abs=1e-15), (Te, T, K, kind)
    # r* prices the coupon bond at K
    A, B = hw_bond_coeffs(P, f, a, sigma, Tf, 2.0, [3.0, 4.0, 5.0])
    rs = jamshidian_rstar(A, B, [0.04, 0.04, 1.04], 1.0)
    assert sum(c * Aj * math.exp(-Bj * rs) for c, Aj, Bj in zip([0.04, 0.04, 1.04], A, B)) == pytest.approx(1.0, rel=1e-13)


def test_jamshidian_payer_minus_receiver_is_the_forward_swap(hw):
    from oracle_lib import Oracle
    o = Oracle(**continuous_theta())
    s, _ = o.bond_curve_sums(6, 1 << 12)
    P, f = o.curve_finalize(s, 1 << 12)
    a, sigma, Tf = float(o.p.a), float(o.p.sigma), float(o.p.T_final)
    for Te, tenor, freq, dk in ((1.0, 5.0, 1, 0.0), (2.0, 3.0, 2, 0.01), (4.0, 6.0, 2, -0.01)):
        kappa = par_rate(P, Tf, Te, tenor, freq) + dk
        sw, fl = hw.swaption_schedule(Te, tenor, kappa, freq=freq, notional=1e4)
        Ts, c = flows_of(sw[0], fl)
        pay = swaption_price("payer", P, f, a, sigma, Tf, Te, Ts, c, 1.0, N=1e4)
        rec = swaption_price("receiver", P, f, a, sigma, Tf, Te, Ts, c, 1.0, N=1e4)
        fwd = forward_swap(P, Tf, Te, Ts, c, 1.0, N=1e4)
        assert pay - rec == pytest.approx(fwd, rel=1e-10, abs=1e-9), (Te, tenor, pay, rec, fwd)
        if dk == 0.0:
            # at the money forward payer = receiver, up to the float32 rounding of the coupons (~1e-8 of N)
            assert abs(fwd) < 1e-3 and pay == pytest.approx(rec, rel=1e-5)


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


def test_oracle_book_vs_jamshidian(hw, model):
    o, P, f, P_se = model
    Tf, a, sigma = float(o.p.T_final), float(o.p.a), float(o.p.sigma)
    Te = np.array([1.0, 1.0, 2.0, 3.0, 5.0, 5.0, 7.0])
    ten = np.array([2.0, 5.0, 3.0, 4.0, 5.0, 2.0, 3.0])
    freq = 2
    kappa = [par_rate(P, Tf, t, n, freq) + d for t, n, d in zip(Te, ten, (0.0, 0.01, -0.01, 0.0, 0.005, 0.0, -0.005))]
    kinds = ["payer", "receiver", "payer", "receiver", "payer", "payer", "receiver"]
    sw, fl = hw.swaption_schedule(Te, ten, kappa, freq=freq, notional=100.0, kind=kinds)
    mom = swaption_oracle.swaption_moments(o, 4243, N_SW, sw, fl, P, f)
    cf = np.array(book_closed_form(sw, fl, P, f, a, sigma, Tf))
    up = np.array(book_closed_form(sw, fl, P + P_se, f, a, sigma, Tf))
    dn = np.array(book_closed_form(sw, fl, P - P_se, f, a, sigma, Tf))
    allow = np.abs(up - dn)
    n_mat = len(P)
    cm = np.array([float(s["N"]) * sum(c * interp_mkt(P, T, Tf, n_mat) for T, c in zip(*flows_of(s, fl))) for s in sw])
    for i in range(len(sw)):
        r = pair_algebra(mom[i], N_SW, cm[i])
        assert abs(r["price_cv"] - cf[i]) <= 5 * r["se_cv"] + allow[i], (i, r, cf[i], allow[i])
    r = pair_algebra(mom[-1], N_SW, cm.sum())
    assert abs(r["price_cv"] - cf.sum()) <= 5 * r["se_cv"] + allow.sum(), (r, cf.sum())
    # the book's first moments are the sums over its options
    assert mom[-1][0] == pytest.approx(mom[:-1, 0].sum(), rel=1e-12)
    assert mom[-1][1] == pytest.approx(mom[:-1, 1].sum(), rel=1e-12)
