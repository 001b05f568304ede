"""Jamshidian's closed form for European swaptions (coupon-bond options) under Hull-White (CPU only, no GPU).

A coupon-bond option pays N max(0, s (sum_j c_j P(T_e, T_j) - K)) at T_e.  Under Hull-White P(T_e, T_j) = A_j e^{-B_j r}
with every A_j > 0, B_j > 0, so with c_j > 0 the bond is decreasing in r: solve sum_j c_j A_j e^{-B_j r*} = K, and the
option is the sum of the zero-coupon bond options struck at X_j = A_j e^{-B_j r*} (Jamshidian, 1989)."""
import math

from scipy.optimize import brentq

from cap_closed_form import bond_option, interp_mkt


def hw_bond_coeffs(P_mkt, f_mkt, a, sigma, T_final, Te, Ts):
    """A_j, B_j of P(T_e, T_j) = A_j exp(-B_j r(T_e)) on the market curves (interpolated like interp_mkt), the
    expressions of the engine's bond plan in float64"""
    n = len(P_mkt)
    P0e, f0e = interp_mkt(P_mkt, Te, T_final, n), interp_mkt(f_mkt, Te, T_final, n)
    var = sigma * sigma / (4.0 * a) * (1.0 - math.exp(-2.0 * a * Te))
    A, B = [], []
    for T in Ts:
        b = (1.0 - math.exp(-a * (T - Te))) / a
        A.append(interp_mkt(P_mkt, T, T_final, n) / P0e * math.exp(b * f0e - var * b * b))
        B.append(b)
    return A, B


def jamshidian_rstar(A, B, c, K):
    """the short rate at which the coupon bond sum_j c_j A_j e^{-B_j r} is worth K"""
    def g(r):
        return sum(cj * Aj * math.exp(-Bj * r) for cj, Aj, Bj in zip(c, A, B)) - K
    lo, hi = -0.5, 0.5
    while g(lo) < 0.0:
        lo *= 2.0
    while g(hi) > 0.0:
        hi *= 2.0
    return brentq(g, lo, hi, xtol=1e-15, rtol=1e-15, maxiter=200)


def swaption_price(kind, P_mkt, f_mkt, a, sigma, T_final, Te, Ts, c, K, N=1.0):
    """N x (payer: sum_j c_j ZBP(T_e, T_j, X_j); receiver: the same with ZBC)"""
    A, B = hw_bond_coeffs(P_mkt, f_mkt, a, sigma, T_final, Te, Ts)
    rs = jamshidian_rstar(A, B, c, K)
    n = len(P_mkt)
    P0e = interp_mkt(P_mkt, Te, T_final, n)
    bk = "cap" if kind == "payer" else "floor"
    return N * sum(cj * bond_option(bk, P0e, interp_mkt(P_mkt, T, T_final, n), Aj * math.exp(-Bj * rs), a, sigma, Te, T)
                   for cj, T, Aj, Bj in zip(c, Ts, A, B))


def forward_swap(P_mkt, T_final, Te, Ts, c, K, N=1.0):
    """payer - receiver: N (K P0(T_e) - sum_j c_j P0(T_j))"""
    n = len(P_mkt)
    return N * (K * interp_mkt(P_mkt, Te, T_final, n) - sum(cj * interp_mkt(P_mkt, T, T_final, n) for cj, T in zip(c, Ts)))


def flows_of(sw, flows):
    """(T_j, c_j) lists of one option of a (swaptions, flows) book"""
    rows = flows[int(sw["first_flow"]):int(sw["first_flow"]) + int(sw["n_flows"])]
    return [float(t) for t in rows["T"]], [float(x) for x in rows["c"]]


def book_closed_form(swaptions, flows, P_mkt, f_mkt, a, sigma, T_final):
    """per-option prices of a book (kind per option: 0 payer, 1 receiver)"""
    out = []
    for sw in swaptions:
        Ts, c = flows_of(sw, flows)
        out.append(swaption_price("payer" if int(sw["kind"]) == 0 else "receiver", P_mkt, f_mkt, a, sigma, T_final,
                                  float(sw["T_exercise"]), Ts, c, float(sw["K"]), float(sw["N"])))
    return out


def par_rate(P_mkt, T_final, Te, tenor, freq):
    """the fixed rate of the spot-starting swap from T_e worth zero today"""
    n = len(P_mkt)
    Ts = [Te + k / freq for k in range(1, int(round(tenor * freq)) + 1)]
    ann = sum(interp_mkt(P_mkt, T, T_final, n) for T in Ts) / freq
    return (interp_mkt(P_mkt, Te, T_final, n) - interp_mkt(P_mkt, Ts[-1], T_final, n)) / ann
