"""Hull-White closed forms and the pair-moment algebra shared by the cap / floor tests (CPU only, no GPU)."""
import math

import numpy as np


def continuous_theta(**overrides):
    """model overrides whose theta is continuous at the break (theta_a1 = theta_a0 + (theta_b0 - theta_b1) theta_break),
    so that the central-difference forward curve has no kink there"""
    p = dict(theta_a0=0.012, theta_b0=0.0014, theta_b1=0.001, theta_break=5.0)
    p.update(overrides)
    p["theta_a1"] = float(np.float32(p["theta_a0"] + (p["theta_b0"] - p["theta_b1"]) * p["theta_break"]))
    return p


def interp_mkt(data, T, T_final, n_mat):
    """P_mkt(T) as the engine's interp_mkt evaluates it (float32: index by truncation, one fused multiply-add)"""
    f = np.float32
    data = np.asarray(data, np.float32)
    spacing = f(f(T_final) / f(n_mat - 1))
    inv = f(f(1.0) / spacing)
    T = f(T)
    idx = int(f(T * inv))
    if idx >= n_mat - 1:
        return float(data[n_mat - 1])
    al = f(f(np.float64(idx) * np.float64(-spacing) + np.float64(T)) * inv)
    om = f(f(1.0) - al)
    return float(f(np.float64(data[idx]) * np.float64(om) + np.float64(f(al * data[idx + 1]))))


def Phi(x):
    return 0.5 * math.erfc(-x / math.sqrt(2.0))


def bond_option(kind, P0r, P0p, K, a, sigma, Tr, Tp):
    """ZBP (kind "cap") or ZBC (kind "floor") of a zero-coupon bond: expiry Tr, maturity Tp, strike K"""
    B = (1.0 - math.exp(-a * (Tp - Tr))) / a
    sp = sigma * math.sqrt((1.0 - math.exp(-2.0 * a * Tr)) / (2.0 * a)) * B
    h = math.log(P0p / (K * P0r)) / sp + 0.5 * sp
    if kind == "cap":
        return K * P0r * Phi(sp - h) - P0p * Phi(-h)
    return P0p * Phi(h) - K * P0r * Phi(h - sp)


def strip_closed_form(kind, caps, P_mkt, a, sigma, T_final):
    """per-caplet N * ZBP / ZBC on the market curve P_mkt (interpolated like interp_mkt), and the strip's sum"""
    n_mat = len(P_mkt)
    v = np.array([float(c["N"]) * bond_option(kind, interp_mkt(P_mkt, c["T_reset"], T_final, n_mat),
                                              interp_mkt(P_mkt, c["T_pay"], T_final, n_mat), float(c["K"]), a, sigma,
                                              float(c["T_reset"]), float(c["T_pay"])) for c in caps])
    return v, float(v.sum())


def atm_rate(P_mkt, resets, pays, T_final):
    """par rate of the strip: (P0(T_r, first) - P0(T_p, last)) / sum tau_i P0(T_p, i)"""
    n = len(P_mkt)
    ann = sum((tp - tr) * interp_mkt(P_mkt, tp, T_final, n) for tr, tp in zip(resets, pays))
    return (interp_mkt(P_mkt, resets[0], T_final, n) - interp_mkt(P_mkt, pays[-1], T_final, n)) / ann


def pair_algebra(mom, n_pairs, control_mean):
    """hw1f_cap_result's statistics from five pair moments: n_pairs samples of X/2, Y/2"""
    n = float(n_pairs)
    sx, sy, sxx, syy, sxy = 0.5 * mom[0], 0.5 * mom[1], 0.25 * mom[2], 0.25 * mom[3], 0.25 * mom[4]
    mx, my = sx / n, sy / n
    vxx = max((sxx - sx * mx) / (n - 1), 0.0)
    vyy = max((syy - sy * my) / (n - 1), 0.0)
    cxy = (sxy - sx * my) / (n - 1)
    beta = cxy / vyy if vyy > 0 else 0.0
    vcv = max(vxx - 2 * beta * cxy + beta * beta * vyy, 0.0)
    return {"price_raw": mx, "se_raw": math.sqrt(vxx / n), "price_cv": mx - beta * (my - control_mean),
            "se_cv": math.sqrt(vcv / n), "beta": beta}
