"""Wall time of the book vega (hw1f_swaptions_vega: sigma, sigma - eps, sigma + eps on one set of paths) next to the
pricing call it extends, for a swaption book and a cap strip, and a Q1 bond-curve call on the same paths.

Setup of tools/swaption_bench.py: default model (1000 steps, 101 maturities), 2^20 subsequences, the 45-option ATM payer
grid (expiries 1..9 x tenors 1..(10 - expiry), semi-annual, 330 flows, last exercise step 900) and the 39 quarterly ATM
caplets (last reset step 975).  Blocking calls through the Python layer, warmed, alternated in one process, median of
--reps; both arithmetic modes.  The ratio vega / pricing says what the two bumped scenarios add: in decomposed mode
they share the path stepping and only add payoffs at the exercise steps.  The card's name and power limit are
recorded beside the numbers.

    python tools/book_vega_bench.py [--reps 30] [--out profiles/r05_book_vega_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
sys.path.insert(0, os.path.join(os.getcwd(), "tools"))
import hw1f_b200 as hw  # noqa: E402
from cap_bench import gpu_info  # noqa: E402
from cap_closed_form import atm_rate  # noqa: E402
from swaption_bench import grid_book  # noqa: E402


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--paths", type=int, default=1 << 20)
    ap.add_argument("--eps", type=float, default=1e-3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    n = args.paths
    eng = hw.Engine(device=0)
    curve = eng.bond_curve(hw.Rng(1, n))
    P, f = curve["P"], curve["f"]
    Tf = float(eng.params.T_final)
    sw, fl = grid_book(P, Tf)
    resets = 0.25 * np.arange(1, 40)
    pays = resets + 0.25
    caps = hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, Tf))
    result = {"model": "default (1000 steps, 101 maturities)", "n_paths": n, "eps": args.eps, "n_swaptions": len(sw),
              "n_flows": len(fl), "last_exercise_step": 900, "n_caplets": len(caps), "last_reset_step": 975,
              "reps": args.reps, **gpu_info(), "modes": {}}
    for mode_name, mode in (("decomposed", hw._ffi.MODE_DECOMPOSED), ("reference_order", hw._ffi.MODE_REFERENCE_ORDER)):
        eng.set_mode(mode)
        rng = hw.Rng(2, n)
        fns = {
            "swaptions": lambda: eng.swaptions(rng.seek(0), sw, fl, P, f),
            "swaptions_vega": lambda: eng.swaptions_vega(rng.seek(0), sw, fl, P, f, eps=args.eps),
            "cap_floor_cap": lambda: eng.cap_floor(rng.seek(0), caps, P, f, kind="cap"),
            "cap_floor_vega_cap": lambda: eng.cap_floor_vega(rng.seek(0), caps, P, f, kind="cap", eps=args.eps),
            "bond_curve": lambda: eng.bond_curve(rng.seek(0), timing=False),
        }
        for fn in fns.values():   # warm-up
            for _ in range(3):
                fn()
        eng.synchronize()
        t = {k: [] for k in fns}
        for _ in range(args.reps):   # alternated
            for k, fn in fns.items():
                t[k].append(wall(fn))
        med = {k: float(np.median(v)) for k, v in t.items()}
        spread = {k: [float(np.percentile(v, 10)), float(np.percentile(v, 90))] for k, v in t.items()}
        v = eng.swaptions_vega(rng.seek(0), sw, fl, P, f, eps=args.eps)
        c = eng.cap_floor_vega(rng.seek(0), caps, P, f, kind="cap", eps=args.eps)
        result["modes"][mode_name] = {
            "median_ms": med, "p10_p90_ms": spread, "swaptions_vega_event_ms_last": v["sim_ms"],
            "swaptions_vega_over_swaptions": med["swaptions_vega"] / med["swaptions"],
            "cap_vega_over_cap": med["cap_floor_vega_cap"] / med["cap_floor_cap"],
            "swaptions_vega_over_bond_curve": med["swaptions_vega"] / med["bond_curve"],
            "book_vega": v["book"]["vega"], "book_vega_se": v["book"]["vega_se"],
            "strip_vega": c["strip"]["vega"], "strip_vega_se": c["strip"]["vega_se"],
        }
        print(mode_name, json.dumps(result["modes"][mode_name]))
    eng.close()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
