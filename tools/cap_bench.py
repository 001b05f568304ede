"""Wall time of a cap / floor strip priced in one pass (hw1f_cap_floor) next to a Q1 bond-curve call (hw1f_bond_curve) on the
same paths, and next to what a user without the strip call does today for a floor: hw1f_zbc_cv once per reset date.

Default model (1000 steps, 101 maturities), 2^20 subsequences, 39 quarterly ATM caplets (resets 0.25 .. 9.75, last reset
step 975).  Blocking calls through the Python layer (host buffers in and out), warmed, alternated in one process, median
of --reps; both arithmetic modes.  The card's name and power limit are recorded beside the numbers.

    python tools/cap_bench.py [--reps 30] [--out r03_cap_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.getcwd())
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import hw1f_b200 as hw  # noqa: E402
from cap_closed_form import atm_rate  # noqa: E402


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, power = [s.strip() for s in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as exc:   # no nvidia-smi: the device name from the runtime, power limit unknown
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unknown ({exc.__class__.__name__})"}


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
    resets = 0.25 * np.arange(1, 40)
    pays = resets + 0.25
    caps = hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, float(eng.params.T_final)))
    steps = [int(round(float(np.float32(t)) / float(eng.constants.dt))) for t in caps["T_reset"]]
    result = {"model": "default (1000 steps, 101 maturities)", "n_paths": n, "n_caplets": len(caps),
              "last_reset_step": steps[-1], "reps": args.reps, **gpu_info(), "modes": {}}
    for mode_name, mode in (("decomposed", hw._ffi.MODE_DECOMPOSED), ("reference_order", hw._ffi.MODE_REFERENCE_ORDER)):
        eng.set_mode(mode)
        rng = hw.Rng(2, n)

        def cap():
            eng.cap_floor(rng.seek(0), caps, P, f, kind="cap")

        def floor():
            eng.cap_floor(rng.seek(0), caps, P, f, kind="floor")

        def q1():
            eng.bond_curve(rng.seek(0), timing=False)

        def zbc_per_reset():   # a floor priced the way the engine allowed before: one ZBC call per reset date
            for c, k in zip(caps, steps):
                eng.zbc_cv(rng.seek(0), P, f, S1=float(c["T_reset"]), S2=float(c["T_pay"]), K=float(c["K"]), n_steps_S1=k)

        fns = {"cap_floor_cap": cap, "cap_floor_floor": floor, "bond_curve": q1, "zbc_cv_per_reset": zbc_per_reset}
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
        sim = eng.cap_floor(rng.seek(0), caps, P, f, kind="cap")["sim_ms"]
        result["modes"][mode_name] = {
            "median_ms": med, "p10_p90_ms": spread, "cap_event_ms_last": sim,
            "cap_over_bond_curve": med["cap_floor_cap"] / med["bond_curve"],
            "zbc_per_reset_over_cap_floor": med["zbc_cv_per_reset"] / med["cap_floor_floor"],
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
