#!/usr/bin/env python
"""bench.py -- HW1F path-steps/s on the BASELINE.json headline workload.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch: the Q1 bond-curve workload of
BASELINE.json (`configs[0]`, the configuration the metric is quoted on): 2^20 RNG subsequences x 2
antithetic paths x 1000 exact-discretisation steps per GPU, stateless XORWOW seeding included,
deterministic two-level reduction to 202 double moments.  With N > 1 every rank simulates its own
disjoint subsequence range (weak scaling) and the moment vectors are combined with ONE NCCL
all-reduce of 202 doubles per step.

`value`  : device-timed (CUDA events on the launching stream), nothing crosses PCIe in the region.
`e2e`    : the public host-buffer calls a user makes (set_model H2D + simulate + finalise + D2H of
           P, f, P_se, every step), wall-clock between synchronisations: hw1f_bond_curve_submit / _collect with four
           result slots in flight at N = 1 (`e2e.blocking` = the one-call form, the host waiting after every step).
`roofline`: this path is instruction-issue / FP32+XU pipe bound (SURVEY 8d), not HBM or tensor:
           achieved = algorithmic pipe instructions/s (12 issue slots per path-step), peak = the
           issue rate measured by the engine's own pipe probes on this GPU at the clock seen.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "HW1F path-steps/s (2M antithetic paths, 1000 steps)"
UNIT = "path-steps/s"
N_PATHS_LOG2 = 20          # reference N_PATHS = 1024*1024 (include/common.cuh:16)
# Algorithmic pipe instructions per path-step (DESIGN.md section 4).
#   reference-order arithmetic (SURVEY 8d): 6.75 FP32 + 1.0 MUFU + 3.75 INT + 0.5 I2F = 12 issue slots
#   decomposed arithmetic (default mode)   : 2.25 FP32 + 1.0 MUFU + 3.75 INT + 0.5 I2F = 7.5 issue slots
#     (per Box-Muller pair and lane = 4 path-steps: 4 Box-Muller FP32 + 5 for the two-step recursion; the loop
#      body's SASS is 299 dispatch cycles per 40 path-steps = 7.48)
#   Q1 save points: reference-order mode adds 4 MUFU.EX2 per 40 path-steps (1.1 MUFU per path-step); decomposed
#   mode evaluates 2cosh(z)-2 as a polynomial on the FMA pipe (no XU work)
def workload_string(paths_log2=N_PATHS_LOG2, n_steps=1000, n_mat=101):
    """the same `config.workload` for both arms: the driver compares the two lines' configs"""
    return (f"Q1 bond curve P(0,T), f(0,T): 2^{paths_log2} XORWOW subsequences x 2 antithetic paths x {n_steps} steps "
            f"per GPU, r0=0.012 a=1 sigma=0.1, {n_mat} maturities, seeding included")


# committed `ncu --set full` summaries of the dominant kernel per arithmetic mode (tools/ncu_summary.py)
NCU_CAPTURE = {"decomposed": "profiles/r02_ncu_full_fast_kernel.csv",
               "reference_order": "profiles/r01_ncu_full_bond_curve_v3.csv"}

ALGO = {
    "decomposed": {"issue": 7.5, "fp32": 2.25, "xu": 1.0},
    "reference_order": {"issue": 12.0, "fp32": 6.75, "xu": 1.1},
}


class ClockSampler(threading.Thread):
    """samples SM clock / throttle reasons with NVML while the timed regions run"""

    def __init__(self, index, period_s=0.01):
        super().__init__(daemon=True)
        self.index, self.samples, self._stop, self.period_s = index, [], threading.Event(), period_s
        self.max_mhz, self.ok = None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(
                    nv, "nvmlDeviceGetCurrentClocksEventReasons") else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                power = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                self.samples.append((time.time(), mhz, reasons, power))
            except Exception:
                pass
            time.sleep(self.period_s)

    def stop(self):
        self._stop.set()

    def summary(self, t0, t1):
        sel = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        if not sel:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        bits = 0
        for s in sel:
            bits |= s[2]
        reasons = [n for b, n in names.items() if bits & b and n != "gpu_idle"]
        return {"sm_mhz": statistics.median(s[1] for s in sel), "sm_max_mhz": self.max_mhz, "reasons": reasons,
                "power_w_max": max(s[3] for s in sel), "samples": len(sel)}


def read_json(path):
    try:
        with open(path) as fh:
            return json.load(fh)
    except (OSError, ValueError):
        return {"file": os.path.relpath(path, ROOT), "missing": True}


def read_ncu_capture(rel_path):
    """pipe / issue figures of the dominant kernel from the committed `ncu --set full` summary
    (profiles/*.csv written by tools/ncu_summary.py); nothing is hard-coded here"""
    import csv
    path = os.path.join(ROOT, rel_path)
    if not os.path.exists(path):
        return {"file": rel_path, "missing": True}
    m = {}
    with open(path, newline="") as fh:
        for row in csv.reader(fh):
            if len(row) >= 2 and row[0] != "metric":
                m[row[0]] = row[1]

    def num(key):
        try:
            return float(m[key].replace(",", ""))
        except (KeyError, ValueError):
            return None
    issue = num("smsp__issue_active.avg.pct_of_peak_sustained_active")
    fma_cyc = num("sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active")
    fma_inst = num("sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active")
    pre, suf = "smsp__average_warps_issue_stalled_", "_per_issue_active.ratio"
    stalls = {k[len(pre):-len(suf)]: float(v) for k, v in m.items() if k.startswith(pre) and k.endswith(suf)}
    stalls.pop("selected", None)
    dram = None
    if num("dram__bytes_read.sum") is not None:
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        with open(path, newline="") as fh:
            units = {r[0]: r[2] for r in csv.reader(fh) if len(r) >= 3}
        dram = sum((num(k) or 0.0) * scale.get(units.get(k, "byte"), 1.0)
                   for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
    return {
        "file": rel_path, "source": "committed ncu --set full summary, read at run time (static: not measured in this run)",
        "kernel_name": m.get("Kernel Name", "")[:60],
        "kernel_us": num("gpu__time_duration.sum"),
        "registers": num("launch__registers_per_thread"), "block": num("launch__block_size"),
        "issue_active_pct": issue,
        # packed FP32x2 instructions hold the dispatch port for two cycles: port utilisation =
        # issue-active + (fma-pipe cycles - fma instructions)
        "dispatch_port_pct": (issue + fma_cyc - fma_inst) if None not in (issue, fma_cyc, fma_inst) else None,
        "xu_pipe_pct": num("sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active"),
        "alu_pipe_pct": num("sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active"),
        "fma_pipe_cycles_pct": fma_cyc,
        "top_stall": max(stalls, key=stalls.get) if stalls else None,
        "dram_bytes": dram,
    }


def _wall_ms(fn, steps, warmup, sync):
    for i in range(warmup):
        fn(i)
    sync()
    ts = []
    for i in range(steps):                      # every call returns host results, i.e. it ends synchronised
        t0 = time.perf_counter()
        fn(100 + i)
        ts.append((time.perf_counter() - t0) * 1e3)
    sync()
    return statistics.median(ts)                # one preempted call out of ten moved the mean by 13 % on a shared host


def measure_workloads(eng, hw, n_paths, mkt):
    """the other north-star workloads (BASELINE.json configs[2], configs[3]) through the public host-buffer API
    (wall clock, every call returns host results) next to the reference's own host functions on the SAME GPU in the
    SAME run (oracle/_ref/ref_harness: src/3_sensitivity_analysis.cu:697-834, src/2_option_pricing.cu:210-468,
    src/3:527-654).  Outside every timed region of the headline metric."""
    import tempfile
    P, f = mkt["P"], mkt["f"]
    sync = eng.synchronize
    out = {}

    def add(key, ms, what):
        out[key] = {"engine_ms": ms, "reference_ms": None, "ratio": None, "what": what}

    add("q1_bond_curve", _wall_ms(lambda i: eng.bond_curve(hw.Rng(i, n_paths)), 20, 3, sync),
        "hw1f_bond_curve vs init_rng + simulate_zcb + compute_average_and_forward + D2H")
    add("q2b_zbc_cv", _wall_ms(lambda i: eng.zbc_cv(hw.Rng(i, n_paths), P, f), 20, 3, sync),
        "hw1f_zbc_cv vs init_rng + simulate_ZBC_control_variate + D2H of 5 moments (src/2:107-208)")
    add("q3_pathwise", _wall_ms(lambda i: eng.vega_pathwise(hw.Rng(i, n_paths), P, f), 20, 3, sync),
        "hw1f_vega_pathwise vs init_rng + simulate_sensitivity + D2H (src/3:236-272)")
    add("q3_sequence", _wall_ms(lambda i: eng.vega(hw.Rng(i, n_paths), P, f), 10, 2, sync),
        "hw1f_vega (reference draw windows: pathwise [0,500), CRN FD [500,1000), recalibrated FD [1000,2000)) vs "
        "init_rng + run_sensitivity_mc + run_finite_difference + run_finite_difference_recalibrated (src/3:697-834)")
    add("q3_single_window", _wall_ms(lambda i: eng.fused(hw.Rng(i, n_paths), P, f), 10, 3, sync),
        "hw1f_fused: curve + ZBC/CV + pathwise vega + CRN FD bumps on ONE window of normals (statistically equivalent "
        "to the Q3 sequence, not stream-identical; no reference counterpart)")
    add("zbc_validation_20_seeds",
        _wall_ms(lambda i: eng.zbc_cv_batch([i * 1000003 + r * 12345 for r in range(20)], n_paths, P, f), 5, 1, sync),
        "hw1f_zbc_cv_batch (20 seeds, one launch) vs run_zbc_statistical_validation (src/2:210-468)")
    add("vega_validation_20_seeds",
        _wall_ms(lambda i: eng.vega_pathwise_batch([i * 1000003 + r * 982451653 for r in range(20)], n_paths, P, f),
                 5, 1, sync),
        "hw1f_vega_pathwise_batch (20 seeds, one launch) vs run_statistical_validation (src/3:527-654)")

    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    if not os.path.exists(harness):
        out["reference"] = "oracle/_ref/ref_harness not built: engine times only"
        return out
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    with tempfile.TemporaryDirectory() as td:
        os.makedirs(os.path.join(td, "data"))

        def run(args, key_json):
            o = os.path.join(td, "o.json")
            try:
                subprocess.run([harness] + args + [o], check=True, cwd=td, env=env, stdout=subprocess.DEVNULL,
                               stderr=subprocess.DEVNULL, timeout=600)
                with open(o) as fh:
                    return json.load(fh)[key_json]
            except Exception as exc:   # noqa: BLE001  (a failed reference leg leaves the engine numbers standing)
                print(f"[bench] reference leg {args} failed: {exc}", file=sys.stderr)
                return None
        ref = {
            "q1_bond_curve": run(["bench", "q1", "20", "3"], "workload_ms_per_step"),
            "q2b_zbc_cv": run(["bench", "q2", "20", "3"], "workload_ms_per_step"),
            "q3_pathwise": run(["bench", "q3", "20", "3"], "workload_ms_per_step"),
            "q3_sequence": run(["workload", "q3seq", "10", "2"], "wall_ms_per_step"),
            "zbc_validation_20_seeds": run(["workload", "zbc20", "3", "1"], "wall_ms_per_step"),
            "vega_validation_20_seeds": run(["workload", "vega20", "3", "1"], "wall_ms_per_step"),
        }
    for k, v in ref.items():
        if v is not None:
            out[k]["reference_ms"] = v
            out[k]["ratio"] = v / out[k]["engine_ms"]
    out["note"] = ("engine: median wall ms per public call, host buffers in and out; reference: q1/q2b/q3_pathwise CUDA-event "
                   "time of init_rng + kernel + D2H, the others wall ms of its own host functions (cudaMalloc/cudaFree "
                   "and 50 MB state copies included -- that part varies several-fold between boxes)")
    return out


CLOSED_FORM = {"P_0_5": 0.947126, "P_0_10": 0.859387, "zbc": 0.025255}   # continuous-time HW values, SURVEY 0.1


def scaling_run(eng, hw, torch, dist, dev, stream, rank, world, peer, mkt, total_log2):
    """BASELINE.json configs[4]: 2^30 XORWOW subsequences (2^31 antithetic paths) x 1000 steps, curve + ZBC/control variate
    + antithetic pathwise vega + both CRN FD bumps from ONE fused launch per rank, sharded by contiguous subsequence
    range (strong scaling), ONE all-reduce of 220 doubles, hw1f_fused_finish on every rank.  Device-timed, max over ranks."""
    nm, n_steps = eng.n_mat, eng.n_steps
    total = 1 << total_log2
    first, count = hw.package.parallel.shard_paths(total, rank, world)
    mom = torch.zeros(2 * nm + 18, dtype=torch.float64, device=dev)

    def one_pass(seed):
        eng.fused_moments(hw.Rng(seed, count, first_path=first), mkt["P"], mkt["f"], mom.data_ptr(), eps=0.001,
                          n_steps_S1=500)
        if peer is None and world > 1:     # with the peers attached the kernel's last block has already exchanged
            dist.all_reduce(mom)

    one_pass(20251019)          # builds the seed-independent jump tables of this shard (untimed)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    one_pass(20251018)
    e1.record()
    torch.cuda.synchronize()
    secs = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(secs, op=dist.ReduceOp.MAX)
    res = eng.fused_finish(mom.data_ptr(), total, float(mkt["P"][-1]), eps=0.001, n_steps_S1=500)
    z, v = res["zbc"], res["vega"]
    s = float(secs.item())
    return {
        "workload": f"configs[4]: fused curve + ZBC/CV + antithetic pathwise vega + CRN FD bumps, 2^{total_log2} "
                    f"subsequences x 2 antithetic x {n_steps} steps, ONE launch per rank + one all-reduce of "
                    f"{2 * nm + 18} doubles", "scaling": "strong", "n_gpus": world, "subsequences_per_gpu": count,
        "seconds": s, "path_steps_per_s": 2.0 * total * n_steps / s,
        "P_0_5": float(res["P"][50]), "P_0_10": float(res["P"][100]), "P_0_10_se": float(res["P_se"][100]),
        "zbc_price_cv": z["price_cv_f64"], "zbc_se_cv": z["se_cv"], "beta": z["beta_f64"],
        "vega_pathwise": v["vega_pathwise_f64"], "vega_pathwise_se": v["vega_pathwise_se"], "vega_fd": v["vega_fd"],
        "closed_form": CLOSED_FORM,
        "note": "estimators must be identical on every GPU count: the shards' union is the single-GPU path set; the "
                "distance from the continuous-time values is the reference scheme's O(dt^2) / grid-interpolation bias "
                "plus the 2^20-path noise of the market curve the option is priced on",
    }


def multi_gpu_check(eng, hw, torch, dist, dev, rank, world, peer, mkt):
    """N > 1: every rank simulates its shard of ONE 2^18-subsequence set, the moment vectors are all-reduced (own NVLink
    peer kernel and NCCL), and every rank also simulates the whole set alone: sums must agree to double rounding.
    Once for the Q1 vector (202 doubles), once for the fused vector (220 doubles)."""
    hwp = hw.package.parallel
    total, seed = 1 << 18, 77001
    first, count = hwp.shard_paths(total, rank, world)
    nm = eng.n_mat
    out = {"set": "2^18 subsequences, seed 77001", "tolerance_fail": 1e-6}

    def rel(a, b):
        return float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())

    if peer is not None:
        peer.attach(False)
    for name, n, sim in (
        ("curve", 2 * nm, lambda r, m: eng.bond_curve_moments(r, m.data_ptr())),
        ("fused", 2 * nm + 18, lambda r, m: eng.fused_moments(r, mkt["P"], mkt["f"], m.data_ptr(), eps=0.001,
                                                                 n_steps_S1=500)),
    ):
        single = torch.zeros(n, dtype=torch.float64, device=dev)
        sim(hw.Rng(seed, total), single)
        shard = torch.zeros(n, dtype=torch.float64, device=dev)
        sim(hw.Rng(seed, count, first_path=first), shard)
        torch.cuda.synchronize()
        via_nccl = shard.clone()
        dist.all_reduce(via_nccl)
        out[name + "_nccl_vs_single_max_rel"] = rel(via_nccl, single)
        if peer is not None:
            via_peer = shard.clone()
            peer.all_reduce(via_peer)                  # the exchange as a launch of its own
            peer.attach(True)
            via_tail = torch.zeros(n, dtype=torch.float64, device=dev)
            sim(hw.Rng(seed, count, first_path=first), via_tail)   # exchanged by the kernel's last block
            peer.attach(False)
            torch.cuda.synchronize()
            out[name + "_peer_vs_single_max_rel"] = rel(via_peer, single)
            out[name + "_tail_vs_single_max_rel"] = rel(via_tail, single)
            out[name + "_tail_vs_nccl_max_rel"] = rel(via_tail, via_nccl)
            out[name + "_tail_bit_identical_to_peer_kernel"] = bool((via_tail == via_peer).all())
    if peer is not None:
        peer.attach(True)
    worst = max(v for k, v in out.items() if k.endswith("_vs_single_max_rel"))
    w = torch.tensor([worst], dtype=torch.float64, device=dev)
    dist.all_reduce(w, op=dist.ReduceOp.MAX)
    out["multi_vs_single_max_rel"] = float(w.item())
    out["ok"] = bool(out["multi_vs_single_max_rel"] <= out["tolerance_fail"])
    return out


def run_reference_arm(args, rank, real_stdout):
    """the reference's own CUDA implementation of the path (the reference has no CPU path), driven
    by oracle/_ref/ref_harness on GPU 0; falls back to the OpenMP oracle port if it was not built"""
    if rank != 0:
        return
    harness = os.path.join(ROOT, "oracle", "_ref", "ref_harness")
    n_paths = 1 << N_PATHS_LOG2
    line = {"metric": METRIC, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_string(),
                       "paths_per_gpu": 2 * n_paths, "n_steps": 1000,
                       "arithmetic": "reference kernels (init_rng + simulate_zcb + compute_average_and_forward), seeds pinned",
                       "l2": "not flushed (the reference re-reads its own 50 MB state array every step)",
                       "parallelism": "single GPU on rank 0 (the reference has no multi-GPU path)"}}
    if os.path.exists(harness):
        import tempfile
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
        with tempfile.TemporaryDirectory() as td:     # the tree may be read-only
            out = os.path.join(td, "ref_bench_q1.json")
            subprocess.run([harness, "bench", "q1", str(args.steps), str(args.warmup), out], check=True, env=env,
                           stdout=subprocess.DEVNULL, timeout=1800)
            with open(out) as f:
                r = json.load(f)
        ms = r["workload_ms_per_step"]
        value = r["path_steps_per_step"] / (ms * 1e-3)
        line.update({"value": value, "ms_per_step": ms, "gpu_launches": 3 * args.steps,
                     "kernel_only": {"value": r["path_steps_per_step"] / (r["kernel_ms_per_step"] * 1e-3),
                                     "ms_per_step": r["kernel_ms_per_step"],
                                     "note": "simulate_zcb alone: the reference's own published metric "
                                             "(src/1_bond_pricing.cu:64-71), init_rng excluded"},
                     "init_rng_ms_per_step": r["init_rng_ms_per_step"],
                     "cpu_baseline": {"value": value, "unit": UNIT, "cores": 0, "kind": "reference",
                                      "sample": "unmodified reference kernels rebuilt for sm_100 (CUDA-only reference, "
                                                "no CPU path): init_rng + simulate_zcb + compute_average_and_forward "
                                                "+ D2H per step on the same B200, CUDA-event timed"},
                     "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    else:
        from oracle_lib import Oracle
        o = Oracle()
        n = 1 << 14
        t0 = time.time()
        for _ in range(max(args.steps, 1)):
            o.bond_curve(1234, n)
        dt = (time.time() - t0) / max(args.steps, 1)
        value = 2.0 * n * 1000 / dt
        line.update({"value": value, "ms_per_step": dt * 1e3, "gpu_launches": 0,
                     "cpu_baseline": {"value": value, "unit": UNIT, "cores": o.max_threads(), "kind": "port",
                                      "sample": "OpenMP oracle, 2^14 pairs x 1000 steps per step"},
                     "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    _emit(line, real_stdout)


def _emit(line, real_stdout):
    os.write(real_stdout, (json.dumps(line) + "\n").encode())


def main():
    # stdout carries exactly ONE JSON line (rank 0): everything libraries print (e.g. NCCL's
    # version banner) is diverted to stderr while the benchmark runs
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--paths-log2", type=int, default=N_PATHS_LOG2, help="subsequences per GPU (default 2^20)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--clock-sample-ms", type=float, default=10.0, help="NVML polling period of the clock sampler thread")
    ap.add_argument("--no-workloads", action="store_true", help="skip the Q2b / Q3 / 20-seed workload block (N = 1)")
    ap.add_argument("--no-scaling-run", action="store_true", help="skip the configs[4] fused 2^30 strong-scaling pass")
    ap.add_argument("--scaling-log2", type=int, default=30, help="total subsequences of the scaling run (default 2^30)")
    ap.add_argument("--ncu-capture", default=None, help="committed ncu summary CSV the roofline object cites")
    ap.add_argument("--collective", default="peer", choices=["peer", "nccl"],
                    help="moment all-reduce for N > 1: own NVLink peer-memory kernel (hw1f_comm_*) or NCCL")
    ap.add_argument("--mode", default="decomposed", choices=["decomposed", "reference_order"],
                    help="simulation arithmetic (include/hw1f.h HW1F_MODE_*); both give the same Gaussians")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last device-timed step computed to DIR/*.npy: the moment vector "
                         "(moments.npy, float64) and the P, f, P_se it finishes to (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "engine":
        ap.error("--dump-outputs writes the engine's outputs (--impl engine)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, real_stdout)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import hw1f_b200 as hw

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the HW1F engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        # a short watchdog: a mismatched collective should fail in minutes, not hang the box
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # a dedicated non-default stream: the engine launches on it, torch events / NCCL see it
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    eng = hw.Engine(device=local_rank, stream=stream.cuda_stream)
    eng.set_mode(hw._ffi.MODE_DECOMPOSED if args.mode == "decomposed" else hw._ffi.MODE_REFERENCE_ORDER)
    n_paths = 1 << args.paths_log2
    n_steps, n_mat = eng.n_steps, eng.n_mat
    first_path = rank * n_paths                       # disjoint XORWOW subsequence ranges per rank
    path_steps_per_step = 2.0 * n_paths * n_steps * world
    moments = torch.zeros(2 * n_mat, dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    # the single collective of the path: 202 doubles.  Default: the engine's own peer-memory kernel over
    # NVLink (rank-ordered, bit-identical on all ranks); NCCL if asked for or if CUDA IPC is unavailable.
    peer, collective = None, "none"
    if world > 1:
        collective = "nccl"
        want_peer = torch.tensor([1 if args.collective == "peer" else 0], device=dev)
        if args.collective == "peer":
            try:
                peer = hw.package.parallel.PeerAllReduce(eng, stream)
            except Exception as exc:                   # noqa: BLE001
                print(f"[rank {rank}] peer all-reduce unavailable ({exc}); using NCCL", file=sys.stderr)
                want_peer[0] = 0
        dist.all_reduce(want_peer, op=dist.ReduceOp.MIN)   # all ranks or none
        if int(want_peer.item()) == 1:
            # attached: the LAST BLOCK of every *_moments simulation kernel posts the reduced vector to the peers'
            # mailboxes and sums the slots in rank order itself -- no launch between reduction and exchange
            collective = "peer_nvlink_in_kernel_tail"
            peer.attach(True)
        elif peer is not None:
            peer.close()
            peer = None

    def reduce_moments():
        if peer is not None:
            return                 # done inside the simulation kernel's tail
        if world > 1:
            dist.all_reduce(moments)

    def device_step(seed):
        rng = hw.Rng(seed, n_paths, first_path=first_path)
        eng.bond_curve_moments(rng, moments.data_ptr())
        reduce_moments()

    def e2e_step(seed):
        eng.set_model(eng.params)                    # compute_constants(): H2D of the model tables
        rng = hw.Rng(seed, n_paths, first_path=first_path)
        if world == 1:
            return eng.bond_curve(rng, timing=False)   # the one-call public API: P, f, P_se land in host buffers
        eng.bond_curve_moments(rng, moments.data_ptr())
        reduce_moments()
        return eng.bond_curve_finish(moments.data_ptr(), n_paths * world)   # D2H of P, f, P_se

    sampler = ClockSampler(local_rank, args.clock_sample_ms * 1e-3)
    sampler.start()

    # ---- warm-up (also builds the jump tables once; they are seed independent) ----
    for i in range(args.warmup):
        device_step(1000 + i)
        flush.zero_()
    barrier()

    # ---- device-timed region: per-step event pairs, L2 flushed between steps ----
    launches0 = eng.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_load0 = time.time()
    for i in range(args.steps):
        ev[i][0].record()
        device_step(5000 + i)
        ev[i][1].record()
        flush.zero_()
    barrier()
    t_load1 = time.time()
    launches = eng.launch_count - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(total_ms.item()) / args.steps
    value = path_steps_per_step / (ms_per_step * 1e-3)

    # what the last timed step computed (seed 5000 + steps - 1, so the same arguments give the same inputs), taken
    # before later steps overwrite the moment vector
    dumped = None
    if args.dump_outputs:
        dumped = {"moments": moments.cpu().numpy()}
        dumped.update(eng.bond_curve_finish(moments.data_ptr(), n_paths * world))

    # ---- end-to-end region: public host-buffer API, wall clock between synchronisations ----
    def timed_e2e(loop):
        loop(2 * hw._ffi.ASYNC_SLOTS, 9000)       # warm-up reaches every result slot (each lane builds its tables once)
        barrier()
        t0 = time.time()
        res = loop(args.steps, 7000)
        barrier()
        secs = torch.tensor([time.time() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(secs, op=dist.ReduceOp.MAX)
        return float(secs.item()) * 1e3 / args.steps, res

    def blocking_loop(n, seed0):
        res = None
        for i in range(n):
            res = e2e_step(seed0 + i)
        return res

    # the same steps through hw1f_bond_curve_submit / _collect with all four result slots in flight (every slot is a lane
    # with its own stream): every step still uploads its model tables (set_model), simulates, and has its P, f, P_se
    # read on the host -- but launch latency and the wake-up of the waiting thread no longer sit between two simulations,
    # and the ramp-up of one call (jump tables, first wave's stream derivation) runs under the drain and the tail of
    # another (single GPU; with N > 1 the moments / finish split above is the public path)
    def submit_collect_loop(n, seed0, depth=hw._ffi.ASYNC_SLOTS):
        res, in_flight = None, 0
        for i in range(n):
            if in_flight == depth:
                res = eng.bond_curve_collect(slot=i % depth)
                in_flight -= 1
            eng.set_model(eng.params)
            eng.bond_curve_submit(hw.Rng(seed0 + i, n_paths, first_path=first_path), slot=i % depth)
            in_flight += 1
        for i in range(n - in_flight, n):                  # the submissions still out, oldest first
            res = eng.bond_curve_collect(slot=i % depth)
        return res

    e2e_blocking_ms, last = timed_e2e(blocking_loop)
    e2e_ms, e2e_api = e2e_blocking_ms, "hw1f_bond_curve (blocking)" if world == 1 else "hw1f_bond_curve_moments + all-reduce + hw1f_bond_curve_finish (blocking)"
    if world == 1:
        e2e_ms, last_sc = timed_e2e(submit_collect_loop)
        e2e_api = (f"hw1f_set_model + hw1f_bond_curve_submit / hw1f_bond_curve_collect, {hw._ffi.ASYNC_SLOTS} result slots "
                   "(lanes) in flight, round robin")
        assert (last_sc["P"] == last["P"]).all() and (last_sc["f"] == last["f"]).all()   # same seed, same bits
    t_load2 = time.time()
    e2e_value = path_steps_per_step / (e2e_ms * 1e-3)
    sampler.stop()
    clocks = sampler.summary(t_load0, t_load2)

    collective_check = None
    if peer is not None:   # the same shard moments: exchanged in the kernel tail vs NCCL (every rank takes part)
        peer.attach(False)
        eng.bond_curve_moments(hw.Rng(424242, n_paths, first_path=first_path), moments.data_ptr())
        via_nccl = moments.clone()
        dist.all_reduce(via_nccl)
        peer.attach(True)
        eng.bond_curve_moments(hw.Rng(424242, n_paths, first_path=first_path), moments.data_ptr())
        torch.cuda.synchronize()
        rel = float(((moments - via_nccl).abs() / (via_nccl.abs() + 1e-300)).max())
        collective_check = {"max_rel_diff_vs_nccl": rel, "timeouts": peer.timeouts()}

    # the same steps in the other arithmetic mode, for transparency (device-timed).  EVERY rank runs
    # this loop: device_step contains the all-reduce
    other = "reference_order" if args.mode == "decomposed" else "decomposed"
    eng.set_mode(hw._ffi.MODE_REFERENCE_ORDER if other == "reference_order" else hw._ffi.MODE_DECOMPOSED)
    for i in range(3):
        device_step(1000 + i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_other = min(args.steps, 50)
    e0.record()
    for i in range(n_other):
        device_step(5000 + i)
    e1.record()
    torch.cuda.synchronize()
    other_ms = e0.elapsed_time(e1) / n_other
    eng.set_mode(hw._ffi.MODE_DECOMPOSED if args.mode == "decomposed" else hw._ffi.MODE_REFERENCE_ORDER)

    # ---- one longer sustained figure: ~1 s of back-to-back steps under one event pair (no flush: the step's only
    # inputs are the 17 KB model tables and the L2-resident jump tables) ----
    n_sus = max(200, int(round(1000.0 / max(ms_per_step, 1e-3))))
    for i in range(3):
        device_step(1000 + i)
    barrier()
    e0.record()
    for i in range(n_sus):
        device_step(30000 + i)
    e1.record()
    torch.cuda.synchronize()
    sus = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(sus, op=dist.ReduceOp.MAX)
    sus_ms = float(sus.item())
    sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                 "value": path_steps_per_step * n_sus / (sus_ms * 1e-3),
                 "note": "back-to-back steps, one event pair, max over ranks, L2 not flushed"}

    # ---- market curve for the option workloads: a prior Q1 at 2^20 subsequences, fixed seed (identical on every rank) ----
    mkt = eng.bond_curve(hw.Rng(1234, 1 << 20))

    # ---- N > 1: sharded moments against the single-GPU moments of the same path set (fails the run above 1e-6) ----
    multi_check = None
    if world > 1:
        multi_check = multi_gpu_check(eng, hw, torch, dist, dev, rank, world, peer, mkt)

    # ---- the other north-star workloads next to the reference's own host functions (N = 1, rank 0) ----
    workloads = None
    if world == 1 and not args.no_workloads:
        workloads = measure_workloads(eng, hw, n_paths, mkt)
        q1 = workloads.get("q1_bond_curve")
        if isinstance(q1, dict) and q1.get("reference_ms"):
            # the same workload through the submission lanes (the e2e region above): model upload, simulation and the
            # host read of P, f, P_se every call, four result slots in flight
            q1["engine_ms_four_slots_in_flight"] = e2e_ms
            q1["ratio_four_slots_in_flight"] = q1["reference_ms"] / e2e_ms

    # ---- BASELINE.json configs[4]: the 2^30 fused strong-scaling run on every N ----
    scal = None
    if not args.no_scaling_run:
        scal = scaling_run(eng, hw, torch, dist, dev, stream, rank, world, peer, mkt, args.scaling_log2)
    peer_timeouts = peer.timeouts() if peer is not None else 0
    if collective_check is not None:
        collective_check["timeouts"] = peer_timeouts

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        if multi_check is not None and not multi_check["ok"]:
            sys.exit(3)
        return

    # ---- roofline denominators measured here: issue rate and pipe rates of this GPU ----
    def rate(which, iters=512):
        ms, n = eng.pipe_probe(which, iters)
        return n / (ms * 1e-3)
    ffma, ffma2, mufu, alu, i2f, mix = rate(0), rate(1), rate(2), rate(3), rate(4, 128), rate(6, 128)
    bm_mix = rate(12)                                             # LG2 : SQRT : SIN : COS = 1 : 1 : 1 : 1, the kernel's MUFU mix
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
    issue_peak_nominal = sm_count * 4 * 32 * sm_mhz * 1e6        # lane-instructions/s at the clock seen
    issue_peak = max(ffma, alu, mix)                              # measured: best single-issue stream
    per_gpu = value / world
    algo = ALGO[args.mode]
    xu_frac = per_gpu * algo["xu"] / mufu
    issue_frac = per_gpu * algo["issue"] / issue_peak
    bound = "xu" if xu_frac >= issue_frac else "issue"
    roofline = {
        # this path is bound by the SFU (XU) pipe and by instruction issue, not by HBM or tensor cores
        # (SURVEY 8d); "achieved"/"peak" are for the binding resource, the other one is given beside it
        "bound": bound,
        "achieved": (per_gpu * algo["xu"] if bound == "xu" else per_gpu * algo["issue"]) / 1e9,
        "peak": (mufu if bound == "xu" else issue_peak) / 1e9,
        "unit": "G MUFU/s (thread-level)" if bound == "xu" else "Ginstr/s (thread-level)",
        "frac": max(xu_frac, issue_frac),
        # dram__bytes_read.sum + dram__bytes_write.sum of one simulation-kernel launch
        # (profiles/r01_ncu_full_*.csv): window tables, L2-resident after first touch
        "traffic": read_ncu_capture(args.ncu_capture or NCU_CAPTURE[args.mode]).get("dram_bytes"),
        "traffic_unit": "bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full "
                        "capture (window tables re-read after the L2 flush; algorithmic bytes are 17 KB in, 1.6 KB out)",
        "peak_source": "measured by hw1f_pipe_probe on this GPU in this run (MUFU.EX2 / FFMA / LOP3 / mixed streams); "
                       "MEASURED_PEAKS.json has no FP32/XU entry (HBM and bf16 tensor only)",
        "mode": args.mode,
        "xu_pipe": {"achieved": per_gpu * algo["xu"] / 1e9, "peak_mufu": mufu / 1e9, "frac": xu_frac},
        "issue": {"achieved": per_gpu * algo["issue"] / 1e9, "peak_measured": issue_peak / 1e9,
                  "peak_nominal_at_clock": issue_peak_nominal / 1e9, "frac": issue_frac},
        "fp32_pipe": {"achieved": per_gpu * algo["fp32"] / 1e9, "peak_ffma": ffma / 1e9,
                      "peak_ffma2_lanes": 2 * ffma2 / 1e9, "frac": per_gpu * algo["fp32"] / max(ffma, 2 * ffma2)},
        "probes_Ginstr_s": {"ffma": ffma / 1e9, "ffma2": ffma2 / 1e9, "mufu_ex2": mufu / 1e9, "lop3_shf": alu / 1e9,
                            "i2fp": i2f / 1e9, "hw1f_mix": mix / 1e9, "mufu_box_muller_mix": bm_mix / 1e9},
        "algorithmic_per_path_step": algo,
        # from the committed ncu --set full summary of this kernel (read from the CSV at run time, not measured in
        # this run): the dispatch port is the co-binding resource -- packed FP32x2 instructions hold it for two cycles
        "ncu_capture": read_ncu_capture(args.ncu_capture or NCU_CAPTURE[args.mode]),
        # static: committed timing ablations of the decomposed step (not measured in this run)
        "ablation": read_json(os.path.join(ROOT, "profiles", "r02_ablation.json")) if args.mode == "decomposed" else None,
        "kernel": ("fast_kernel<1,0,0>" if args.mode == "decomposed" else "bond_curve_kernel<1>") +
                  " (prep_lo_kernel and tail_kernel included in the time)",
        "other_mode": {"mode": other, "ms_per_step": other_ms,
                       "value": path_steps_per_step / world / (other_ms * 1e-3),
                       "issue_frac": path_steps_per_step / world / (other_ms * 1e-3) * ALGO[other]["issue"] / issue_peak},
    }

    # ---- steady state of the simulation kernel: time per wave of resident blocks, from two grids that are exact
    # multiples of the resident capacity (launch ramp, seeding launch, reduction and the ragged last wave cancel) ----
    steady = None
    try:
        cap = sm_count * 2                                   # resident 512-thread blocks = chunks of 1024 subsequences
        t_by_waves = {}
        for waves in (4, 8):
            nn = cap * waves * 1024
            ms = sorted(eng.bond_curve(hw.Rng(600 + i, nn))["sim_ms"] for i in range(7))[1:-1]
            t_by_waves[waves] = sum(ms) / len(ms)
        per_wave_ms = (t_by_waves[8] - t_by_waves[4]) / 4.0
        ss_rate = cap * 1024 * 2.0 * n_steps / (per_wave_ms * 1e-3)
        steady = {"ms_per_wave": per_wave_ms, "chunks_per_wave": cap, "value": ss_rate,
                  "xu_frac": ss_rate * algo["xu"] / mufu, "fixed_ms_per_call": t_by_waves[4] - 4.0 * per_wave_ms,
                  "note": "event-timed hw1f_bond_curve at 4 and 8 full waves of resident blocks; the difference is four "
                          "waves of pure simulation (stream derivation and block partials included), the remainder the "
                          "per-call fixed time (prep_lo_kernel, launch ramp, ragged drain, tail_kernel)"}
    except Exception as exc:   # noqa: BLE001
        steady = {"error": str(exc)}
    roofline["steady_state"] = steady
    # the same fraction for the end-to-end figure: with all result slots in flight the fixed part of one call runs under
    # the simulation of another, so the public API gets closer to the steady-state rate than a lone call can
    if roofline.get("xu_pipe", {}).get("peak_mufu"):
        roofline["end_to_end"] = {"value": e2e_value, "ms_per_step": e2e_ms,
                                  "xu_frac": e2e_value * ALGO[args.mode]["xu"] / 1e9 / roofline["xu_pipe"]["peak_mufu"],
                                  "api": e2e_api}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle_lib import Oracle
        o = Oracle()
        # bounded sample of the same workload sized for ~10 s of wall time on this box's cores
        # (BASELINE.json configs[0] runs the oracle at 2^16; more cores -> a bigger sample)
        t0 = time.time()
        o.bond_curve(1, 1 << 14)
        t_cal = max(time.time() - t0, 1e-3)
        lg = 14
        while lg < 22 and t_cal * (1 << (lg + 1 - 14)) < 12.0:
            lg += 1
        n_cpu = 1 << max(lg, 16)
        t0 = time.time()
        o.bond_curve(1234, n_cpu)
        dt = time.time() - t0
        cpu_baseline = {"value": 2.0 * n_cpu * n_steps / dt, "unit": UNIT, "cores": o.max_threads(), "kind": "port",
                        "sample": f"OpenMP C oracle (oracle/hw1f_oracle.c), Q1 at 2^{n_cpu.bit_length() - 1} "
                                  f"subsequences x 2 x 1000 steps, {dt:.2f} s wall"}

    bad = {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clocks.get("reasons", []))
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.paths_log2, n_steps, n_mat), "arithmetic": args.mode,
                   "paths_per_gpu": 2 * n_paths, "n_steps": n_steps, "l2": "flushed between steps (256 MiB memset, "
                   "outside the per-step event pairs)", "parallelism": (f"path-range sharding x{world}, one all-reduce of 202 doubles per step "
                                                           f"({collective})") if world > 1 else "single GPU"},
        "collective": {"kind": collective, "check": collective_check},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "api": e2e_api,
                "blocking": {"value": path_steps_per_step / (e2e_blocking_ms * 1e-3), "ms_per_step": e2e_blocking_ms,
                             "note": "one call at a time: the host waits for every step before it issues the next"},
                # set_model uploads ONE arena: 2 duplicated drift tables + centring + exp(-Im), 256-byte aligned pieces
                # (with the result slots in flight the lane that runs a step uploads it again: slot 0 is the caller's own
                # upload, the other lanes follow it -> (2 S - 1) / S uploads per step on average over S slots)
                "h2d_bytes_per_step": int((2 * (((n_steps + 2) * 8 + 255) // 256 * 256) + 2 * ((n_mat * 4 + 255) // 256 * 256))
                                          * ((2 * hw._ffi.ASYNC_SLOTS - 1) / hw._ffi.ASYNC_SLOTS if world == 1 else 1)),
                "d2h_bytes_per_step": 3 * n_mat * 4},
        "gpu_launches": int(launches),
        "clocks": clocks, "clock_check": "rejected: thermal/hw slowdown seen" if bad else "ok",
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
        "sustained": sustained,
        "workloads": workloads,
        "scaling_run": scal,
        "check": {"P_0_10": float(last["P"][-1]), "f_0_0": float(last["f"][0]),
                  "multi_vs_single_max_rel": multi_check["multi_vs_single_max_rel"] if multi_check else None,
                  "multi_gpu": multi_check},
        "published_v100_path_steps_per_s": 3.91e11,
    }
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    _emit(line, real_stdout)
    if world > 1:
        dist.destroy_process_group()
    if multi_check is not None and not multi_check["ok"]:
        print(f"[bench] multi-GPU moments differ from the single-GPU moments: {multi_check}", file=sys.stderr)
        sys.exit(3)
    if peer_timeouts:
        print(f"[bench] peer all-reduce timed out {peer_timeouts} times", file=sys.stderr)
        sys.exit(4)


if __name__ == "__main__":
    main()
