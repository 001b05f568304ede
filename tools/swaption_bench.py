"""Wall time of a swaption book priced in one pass (hw1f_swaptions) next to a Q1 bond-curve call (hw1f_bond_curve) and the
39-caplet cap strip (hw1f_cap_floor) on the same paths.

Default model (1000 steps, 101 maturities), 2^20 subsequences.  The book is the ATM payer grid of expiries 1..9 years x
tenors 1..(10 - expiry) years with semi-annual coupons: 45 swaptions, 330 flows, last exercise step 900.  The cap is
tools/cap_bench.py's: 39 quarterly ATM caplets, last reset step 975.  Blocking calls through the Python layer (host
buffers in and out), warmed, alternated in one process, median of --reps; both arithmetic modes.  The card's name and
power limit are recorded beside the numbers.

    python tools/swaption_bench.py [--reps 30] [--out r04_swaption_bench.json]
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
from swaption_closed_form import par_rate  # noqa: E402


def grid_book(P, T_final):
    Te = [e for e in range(1, 10) for _ in range(1, 11 - e)]
    ten = [t for e in range(1, 10) for t in range(1, 11 - e)]
    kappa = [par_rate(P, T_final, e, t, 2) for e, t in zip(Te, ten)]
    return hw.swaption_schedule(Te, ten, kappa, freq=2, kind="payer")


def wall(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--paths", type=int, default=1 << 20)
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
    result = {"model": "default (1000 steps, 101 maturities)", "n_paths": n, "n_swaptions": len(sw),
              "n_flows": len(fl), "last_exercise_step": 900, "n_caplets": len(caps), "last_reset_step": 975,
              "reps": args.reps, **gpu_info(), "modes": {}}
    for mode_name, mode in (("decomposed", hw._ffi.MODE_DECOMPOSED), ("reference_order", hw._ffi.MODE_REFERENCE_ORDER)):
        eng.set_mode(mode)
        rng = hw.Rng(2, n)

        def swaptions():
            eng.swaptions(rng.seek(0), sw, fl, P, f)

        def cap():
            eng.cap_floor(rng.seek(0), caps, P, f, kind="cap")

        def q1():
            eng.bond_curve(rng.seek(0), timing=False)

        fns = {"swaptions": swaptions, "cap_floor_cap": cap, "bond_curve": q1}
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
        res = eng.swaptions(rng.seek(0), sw, fl, P, f)
        result["modes"][mode_name] = {
            "median_ms": med, "p10_p90_ms": spread, "swaptions_event_ms_last": res["sim_ms"],
            "swaptions_over_bond_curve": med["swaptions"] / med["bond_curve"],
            "swaptions_over_cap": med["swaptions"] / med["cap_floor_cap"],
            "book_price_cv": res["book"]["price_cv"], "book_se_cv": res["book"]["se_cv"],
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
