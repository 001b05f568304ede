import sys, os
sys.path.insert(0, os.getcwd())
import numpy as np
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import hw1f_b200 as hw
from oracle_lib import Oracle
import cap_oracle
import swaption_oracle


def cap_strip(eng):
    """four caplets at explicit reset steps (a fifth, two, three and four fifths of the horizon) paying half-way to T_final"""
    dt, Tf = float(eng.constants.dt), float(eng.params.T_final)
    ks = sorted({max(1, round(eng.n_steps * j / 5)) for j in (1, 2, 3, 4)} - {eng.n_steps})
    rows = [(np.float32(k * dt), np.float32(k * dt + 0.5 * (Tf - k * dt)), 0.99, 1.0, k, 0) for k in ks]
    return np.array(rows, [("T_reset", "f4"), ("T_pay", "f4"), ("K", "f4"), ("N", "f4"), ("n_steps_reset", "i4"), ("reserved", "i4")])


def cap_vs_oracle(eng, over, n, c):
    caps = cap_strip(eng)
    got = eng.cap_floor(hw.Rng(6, n), caps, c["P"], c["f"], kind="floor")
    ref = cap_oracle.cap_moments(Oracle(**over), 6, n, caps, c["P"], c["f"], kind="floor")
    mom = np.vstack([got["mom"], np.asarray(got["strip"]["mom"])[None, :]])
    return {"strip_price_cv": got["strip"]["price_cv"], "worst_rel_vs_oracle": float(np.abs(mom / ref - 1).max())}


def swaption_book(eng):
    """a payer and a receiver exercised at a fifth and three fifths of the horizon, on two and three flows up to T_final"""
    dt, Tf, ns = float(eng.constants.dt), float(eng.params.T_final), eng.n_steps
    k1, k2 = max(1, round(ns / 5)), max(1, round(3 * ns / 5))
    T1, T2 = np.float32(k1 * dt), np.float32(k2 * dt)
    flows = np.array([(T1 + 0.5 * (Tf - T1), 0.02), (Tf, 1.02), (T2 + (Tf - T2) / 3, 0.01), (T2 + 2 * (Tf - T2) / 3, 0.01),
                      (Tf, 1.01)], [("T", "f4"), ("c", "f4")])
    sw = np.array([(T1, 1.0, 1.0, 0, k1, 0, 2, 0), (T2, 1.0, 1.0, 1, k2, 2, 3, 0)],
                  [("T_exercise", "f4"), ("K", "f4"), ("N", "f4"), ("kind", "i4"), ("n_steps_exercise", "i4"),
                   ("first_flow", "i4"), ("n_flows", "i4"), ("reserved", "i4")])
    return sw, flows


def swaption_vs_oracle(eng, over, n, c):
    sw, fl = swaption_book(eng)
    got = eng.swaptions(hw.Rng(7, n), sw, fl, c["P"], c["f"])
    ref = swaption_oracle.swaption_moments(Oracle(**over), 7, n, sw, fl, c["P"], c["f"])
    mom = np.vstack([got["mom"], np.asarray(got["book"]["mom"])[None, :]])
    return {"book_price_cv": got["book"]["price_cv"], "worst_rel_vs_oracle": float(np.abs(mom / ref - 1).max())}


for over in (dict(n_steps=8184, n_mat=1024), dict(n_steps=1023, n_mat=1024, T_final=10.23), dict(n_steps=2, n_mat=3, T_final=0.5), dict(n_steps=8192, n_mat=513)):
  for mode in (0, 1):
    eng = hw.Engine(device=0, params=hw.default_params(**over)); eng.set_mode(mode)
    n = (1 << 13) + 5
    c = eng.bond_curve(hw.Rng(1, n))
    S1, S2 = 0.5 * eng.params.T_final, eng.params.T_final
    ns = eng.steps_to(S1)
    print(over, mode, "ns", ns, "P_end", c["P"][-1])
    for name, fn in (("zbc", lambda: eng.zbc_cv(hw.Rng(2, n), c["P"], c["f"], S1=S1, S2=S2, n_steps_S1=ns)["price_cv"]),
                     ("vega", lambda: {k: v for k, v in eng.vega(hw.Rng(3, n), c["P"], c["f"], S1=S1, S2=S2, n_steps_S1=ns).items() if k.startswith("vega") and not k.endswith("se")}),
                     ("fd_recal", lambda: eng.vega_fd_recalibrated(hw.Rng(3, n), S1=S1, S2=S2, n_steps_S1=ns)["vega_fd_recal"]),
                     ("fused", lambda: eng.fused(hw.Rng(4, n), c["P"], c["f"], S1=S1, S2=S2, n_steps_S1=ns)["vega"]["vega_fd"]),
                     ("ci", lambda: float(eng.bond_curve_ci()["f_se"].max())),
                     ("batch", lambda: eng.zbc_cv_batch([1, 2], n, c["P"], c["f"], S1=S1, S2=S2, n_steps_S1=ns)[0][0]),
                     ("cap_floor", lambda: cap_vs_oracle(eng, over, n, c)),
                     ("swaptions", lambda: swaption_vs_oracle(eng, over, n, c)),
                     ("paths", lambda: eng.sample_paths(hw.Rng(5, n), 4).shape)):
        try:
            print("   ", name, fn())
        except Exception as e:
            print("   ", name, "ERR", str(e)[:160])
    eng.close()
