"""Every pricing kernel, pair by pair, against the double-precision evaluation of the same discrete scheme
(tests/f64_reference.py), in both arithmetic modes.

With n_paths = 1 the moments a kernel returns are the summands of one antithetic pair, so a single pair can be compared
with the f64 reference under pair_bound (f64_reference.rel_bound: operation counts plus a MUFU allowance; derived and
checked against the float oracle in tests/test_f64_reference.py).  The first paths cover both float2 lanes (path mod 1024
below / above 512) and both half-warps (path mod 32 below / above 16) of derive_streams, the first and last subsequence
of a chunk, and an index >= 2^32; normal offsets 0 and odd (the cached cos half) where the entry point takes them.
Windows of 33 and 1025 pairs from an odd first path compare the moments with the f64 sums under the summed bounds.

Drift: the default, continuous-theta, 8184 x 1024 and 2 x 3 models use the exact drift integrals.  The a / sigma sweep
compares with the engine's own drift table (the reference's float expressions, whose error at small a dt
test_f64_reference.test_float_drift_table_error measures), so that it measures the kernels' path arithmetic; the gap to
the exact-drift reference is printed beside it.
"""
import numpy as np
import pytest
import torch

from cap_closed_form import continuous_theta
from f64_reference import F64, atm_book, book_rel, caplet_book, pair_bound, rel_bound
from oracle_lib import Oracle

pytestmark = pytest.mark.gpu

SEED = 97
FIRST_PATHS = [0, 17, 515, 1023, (1 << 32) + 530]     # lane A low half, A high half, lane B, last of a chunk, >= 2^32

MODELS = {
    "default": dict(),
    "continuous_theta": continuous_theta(),
    "8184x1024": dict(n_steps=8184, n_mat=1024, T_final=8.184),
    "2x3": dict(n_steps=2, n_mat=3, T_final=0.5),
}
# the a / sigma sweep on 1000 x 101, and two points on the longest grid (8184 steps, dt = 0.001) either side of the
# decomposed mode's limit n_steps dt sig_st / (1 - e^{-a dt}) <= 250 (include/hw1f.h): 233 and 1810
LONG = dict(n_steps=8184, n_mat=1024, T_final=8.184)
SWEEP = ([dict(a=a, sigma=s) for a in (1.0, 0.1, 0.05, 0.01, 0.001) for s in (0.01, 0.1)] +
         [dict(a=0.05, sigma=0.045, **LONG), dict(a=0.01, sigma=0.07, **LONG)])
DECOMP_LIMIT = 250.0


def refused(hw, engine, F):
    """the decomposed mode's accuracy domain (hw1f_api.cu: require_model_sim)"""
    return (engine.mode == hw._ffi.MODE_DECOMPOSED and
            F.n_steps * F.dt * F.sig_st() / (1 - F.e) > DECOMP_LIMIT)


class Setup:
    def __init__(self, hw, engine, over, table=False):
        self.o = Oracle(**over)
        self.F = F64(self.o)
        self.eng = hw.Engine(device=0, params=hw.default_params(**over))
        self.eng.set_mode(engine.mode)
        self.hw = hw
        self.P, self.f = self.o.bond_curve(SEED, 1 << 10)
        self.drift = self.eng.drift_table(0).astype(np.float64) if table else None
        self.exact = not table

    def close(self):
        self.eng.close()


def dev(n):
    return torch.zeros(n, dtype=torch.float64, device="cuda")


def read(S, m):
    """the moments of an asynchronous *_moments call, once the engine's stream has written them"""
    S.eng.synchronize()
    return m.cpu().numpy()


def report(what, gap, bound, extra=""):
    r = float(np.max(gap / bound))
    print(f"{what}: worst |gpu - f64| / pair_bound {r:.3g}{extra}")
    assert np.isfinite(gap).all() and r <= 1.0, (what, r)
    return r


def check_curve(S, first, offset, n_pairs=1):
    F = S.F
    m = dev(2 * F.n_mat)
    S.eng.bond_curve_moments(S.hw.Rng(SEED, n_pairs, first_path=first).seek(offset), m.data_ptr())
    got = read(S, m)[1:F.n_mat]
    steps = np.arange(1, F.n_mat) * F.stride
    st = F.states(SEED, n_pairs, steps, first, offset, drift=S.drift)
    p0 = np.exp(-st[:, :, 2]) + np.exp(-st[:, :, 3])
    Iabs = np.maximum(np.abs(st[:, :, 2]), np.abs(st[:, :, 3]))
    rel = rel_bound(steps, Iabs, np.array([F.sd_I(k * F.dt) for k in steps]))
    return report(f"curve first {first} offset {offset} n {n_pairs}", np.abs(got - p0.sum(0)),
                  pair_bound(p0, rel).sum(0))


def zbc_ref(S, first, offset, n_pairs, n):
    F = S.F
    S1 = float(np.float32(n * np.float32(F.dt)))
    z = F.zbc(SEED, n_pairs, S.P, S.f, n, S1=S1, S2=F.T_final, first_path=first, offset=offset, drift=S.drift)
    rel = rel_bound(n, z["I_abs"].max(1), F.sd_I(S1), r_abs=z["r_abs"].max(1), B=z["B"], sd_r=F.sd_r(S1))
    return S1, z, rel


def check_zbc(S, first, offset, n_pairs=1):
    F = S.F
    n = max(1, F.n_steps // 2)
    S1, z, rel = zbc_ref(S, first, offset, n_pairs, n)
    m = dev(5)
    S.eng.zbc_cv_moments(S.hw.Rng(SEED, n_pairs, first_path=first).seek(offset), S.P, S.f, m.data_ptr(), S1=S1,
                         S2=F.T_final, n_steps_S1=n)
    got = read(S, m)
    X, Y = z["x"].sum(1), z["y"].sum(1)
    ref = np.array([X.sum(), Y.sum()])
    bound = np.array([pair_bound(X, rel, Y).sum(), pair_bound(Y, rel).sum()])
    extra = ""
    if not S.exact:
        Se = Setup.__new__(Setup)
        Se.__dict__.update(S.__dict__, drift=None)
        _, ze, _ = zbc_ref(Se, first, offset, n_pairs, n)
        extra = f"; gap to the exact-drift reference / its value {abs(got[1] / ze['y'].sum() - 1):.3g}"
    return report(f"zbc first {first} offset {offset} n {n_pairs}", np.abs(got[:2] - ref), bound, extra)


def check_pathwise(S, first, offset, n_pairs=1):
    F = S.F
    n = max(1, F.n_steps // 2)
    S1 = float(np.float32(n * np.float32(F.dt)))
    m = dev(2)
    S.eng.vega_pathwise_moments(S.hw.Rng(SEED, n_pairs, first_path=first).seek(offset), S.P, S.f, m.data_ptr(), S1=S1,
                                S2=F.T_final, n_steps_S1=n)
    got = read(S, m)[0]
    pw = F.pathwise(SEED, n_pairs, S.P, S.f, n, S1=S1, S2=F.T_final, first_path=first, offset=offset)
    z = pw["zbc"]
    rel = rel_bound(n, z["I_abs"][:, 0], F.sd_I(S1), r_abs=z["r_abs"][:, 0], B=z["B"], sd_r=F.sd_r(S1))
    # smooth parts, and the whole first term for a pair whose indicator P > K is within the bound of the kink
    kink = np.abs(z["P"][:, 0] - Oracle.K_DEFAULT) <= rel * z["P"][:, 0]
    bound = (pair_bound(pw["term1"][:, 0], rel) + pair_bound(pw["term2"][:, 0], rel, z["y"][:, 0] * np.abs(pw["J"][:, 0]))
             + np.where(kink, np.abs(pw["term1"][:, 0]), 0.0))
    return report(f"pathwise first {first} offset {offset} n {n_pairs}", abs(got - pw["v"][:, 0].sum()),
                  bound.sum() + 1e-12)


def books(S, big=True):
    F = S.F
    k = F.n_steps
    if k < 20:
        cap = caplet_book(F, S.P, [1, 1], 1)
        sw = atm_book(F, S.P, [1, 1], [1, 1], [0, 1])
        return [("cap", cap), ("book", sw)]
    cap = caplet_book(F, S.P, [k // 40, k // 10, k // 10, k // 4, k // 2, 3 * k // 4, k - k // 40], max(1, k // 40))
    sw = atm_book(F, S.P, [k // 10, k // 10, 3 * k // 10, k // 2, k // 2, 7 * k // 10],
                  [k // 20, k // 10, k // 40, k // 10, k // 20, k // 10], [0, 1, 0, 1, 0, 1], big_flows=2048 if big else 0)
    return [("cap", cap), ("book", sw)]


def check_book(S, first, offset, n_pairs=1, vega=False):
    F = S.F
    out = []
    for name, (sw, fl) in books(S, big=not vega):
        bk = F.book(SEED, n_pairs, sw, fl, S.P, S.f, first_path=first, offset=offset, drift=S.drift)
        rel = book_rel(F, bk, sw)
        rng = S.hw.Rng(SEED, n_pairs, first_path=first).seek(offset)
        if not vega:
            if name == "cap":    # the strip kernel (hw1f_cap_floor), not the book kernel
                caps = np.zeros(len(sw), [("T_reset", np.float32), ("T_pay", np.float32), ("K", np.float32),
                                          ("N", np.float32), ("n_steps_reset", np.int32)])
                caps["T_reset"], caps["T_pay"], caps["K"], caps["N"] = sw["T_exercise"], fl["T"], sw["K"], sw["N"]
                caps["n_steps_reset"] = sw["step"]
                res = S.eng.cap_floor(rng, caps, S.P, S.f, kind="cap")
                res["book"] = res.pop("strip")
            else:
                res = S.eng.swaptions(rng, sw, fl, S.P, S.f)
            mom = np.vstack([res["mom"], np.asarray(res["book"]["mom"])[None]])
            got = mom[:, :2]
            ref = np.stack([bk["X"].sum(0), bk["Y"].sum(0)], axis=1)
            bound = np.stack([pair_bound(bk["X"], rel, bk["Y"]).sum(0), pair_bound(bk["Y"], rel).sum(0)], axis=1)
            out.append(report(f"{name} first {first} offset {offset} n {n_pairs}", np.abs(got - ref), bound + 1e-300))
        else:
            eps = 1e-3
            res = S.eng.swaptions_vega(rng, sw, fl, S.P, S.f, eps=eps)
            vm = np.vstack([res["vega_mom"], np.asarray(res["book"]["vega_mom"])[None]])
            bv = F.book_vega(SEED, n_pairs, sw, fl, S.P, S.f, eps, first_path=first, offset=offset)
            bm = pair_bound(bv["Xm"], rel, bv["minus"]["Y"])
            bp = pair_bound(bv["Xp"], rel, bv["plus"]["Y"])
            got = vm[:, [0, 2, 4]]
            ref = np.stack([bv["Xm"].sum(0), bv["Xp"].sum(0), bv["D"].sum(0)], axis=1)
            bound = np.stack([bm.sum(0), bp.sum(0), (bm + bp).sum(0)], axis=1)
            out.append(report(f"{name} vega first {first} offset {offset} n {n_pairs}", np.abs(got - ref),
                              bound + 1e-300))
    return max(out)


@pytest.fixture(scope="module", params=list(MODELS))
def model(request, hw, engine):
    S = Setup(hw, engine, MODELS[request.param])
    yield S
    S.close()


# ---------------------------------------------------------------- single pairs
@pytest.mark.parametrize("first", FIRST_PATHS)
def test_single_pairs(model, first):
    for off in (0, 2):
        check_curve(model, first, off)
    for off in (0, 1):
        check_zbc(model, first, off)
        if model.exact:
            check_pathwise(model, first, off)
        check_book(model, first, off)
        if model.exact and model.F.n_steps == 1000:
            check_book(model, first, off, vega=True)


def test_fused_fd_single_pairs(hw, engine):
    """hw1f_fused_fd_moments (curve, ZBC, pathwise of both twins and the FD bumps of hw1f_vega_fd on one pass), every
    slot per pair against f64 at even offsets 0 and 2 (the fused pass starts on a Box-Muller pair): the curve sums, ZBC X
    and Y, sum (v1 + v2) and sum v1 of the pathwise block, and X-, X+ of the FD scenarios (shifted drift with fd_theta_a1)"""
    S = Setup(hw, engine, {})
    try:
        F, eps, n = S.F, 1e-3, 500
        S1 = float(np.float32(n * np.float32(F.dt)))
        nq, c0 = 2 * F.n_mat + 18, 2 * F.n_mat
        K = Oracle.K_DEFAULT
        for first in FIRST_PATHS:
            for off in (0, 2):
                m = dev(nq)
                S.eng.fused_moments(S.hw.Rng(SEED, 1, first_path=first).seek(off), S.P, S.f, m.data_ptr(), eps=eps,
                                    S1=S1, n_steps_S1=n)
                got = read(S, m)
                what = f"fused first {first} offset {off}"
                # curve slots [1, n_mat): sum p0
                steps = np.arange(1, F.n_mat) * F.stride
                st = F.states(SEED, 1, steps, first, off)
                p0 = np.exp(-st[:, :, 2]) + np.exp(-st[:, :, 3])
                rel = rel_bound(steps, np.maximum(np.abs(st[:, :, 2]), np.abs(st[:, :, 3])),
                                np.array([F.sd_I(k * F.dt) for k in steps]))
                report(what + " curve", np.abs(got[1:F.n_mat] - p0[0]), pair_bound(p0, rel)[0])
                # ZBC X, Y at S1
                S1_, z, rel = zbc_ref(S, first, off, 1, n)
                X, Y = z["x"].sum(1), z["y"].sum(1)
                report(what + " zbc", np.abs(got[c0:c0 + 2] - [X.sum(), Y.sum()]),
                       np.array([pair_bound(X, rel, Y).sum(), pair_bound(Y, rel).sum()]) + 1e-300)
                # pathwise of both twins: sum (v1 + v2), sum v1
                pw = F.pathwise(SEED, 1, S.P, S.f, n, S1=S1, S2=F.T_final, first_path=first, offset=off)
                zz = pw["zbc"]
                b = np.zeros(2)
                for t in range(2):
                    r = rel_bound(n, zz["I_abs"][:, t], F.sd_I(S1), r_abs=zz["r_abs"][:, t], B=zz["B"], sd_r=F.sd_r(S1))
                    kink = np.abs(zz["P"][:, t] - K) <= r * zz["P"][:, t]
                    b[t] = (pair_bound(pw["term1"][:, t], r) + pair_bound(pw["term2"][:, t], r, zz["y"][:, t] *
                            np.abs(pw["J"][:, t])) + np.where(kink, np.abs(pw["term1"][:, t]), 0.0)).sum()
                v = pw["v"][0]
                report(what + " pathwise", np.abs(got[[c0 + 5, c0 + 7]] - [v.sum(), v[0]]),
                       np.array([b.sum(), b[0]]) + 1e-12)
                # FD scenarios sigma -/+ eps
                fd = F.vega_fd(SEED, 1, S.P, S.f, n, eps=eps, S1=S1, first_path=first, offset=off)
                for k, z in enumerate(fd):
                    sg = float(np.float32(F.sigma + (2 * k - 1) * np.float32(eps)))
                    rel = rel_bound(n, z["I_abs"].max(1), F.sd_I(S1, sg), r_abs=z["r_abs"].max(1), B=z["B"],
                                    sd_r=F.sd_r(S1, sg))
                    X, Y = z["x"].sum(1), z["y"].sum(1)
                    base = c0 + 8 + 5 * k
                    report(what + f" FD scenario {k}", np.abs(got[base:base + 2] - [X.sum(), Y.sum()]),
                           np.array([pair_bound(X, rel, Y).sum(), pair_bound(Y, rel).sum()]) + 1e-300)
    finally:
        S.close()


# ---------------------------------------------------------------- windows
@pytest.mark.parametrize("n_pairs", [33, 1025])
def test_windows(model, n_pairs):
    check_curve(model, 7, 0, n_pairs)
    check_zbc(model, 7, 1, n_pairs)
    if model.exact:
        check_pathwise(model, 7, 1, n_pairs)
    check_book(model, 7, 1, n_pairs)


# ---------------------------------------------------------------- a / sigma sweep
@pytest.mark.parametrize("over", SWEEP, ids=lambda o: "-".join(f"{k}{v}" for k, v in o.items()))
def test_sweep(hw, engine, over):
    S = Setup(hw, engine, over, table=True)
    try:
        F = S.F
        tag = f"SWEEP mode {engine.mode} a {over['a']} sigma {over['sigma']} n_steps {F.n_steps}"
        if refused(hw, engine, F):
            # outside the decomposed mode's accuracy domain (include/hw1f.h): refused, never a wrong result
            with pytest.raises(hw.HW1FError, match="decomposed mode is accurate only"):
                check_curve(S, 0, 0)
            print(f"{tag}: refused")
            return
        worst = [check_curve(S, p, 0) for p in FIRST_PATHS[:3]]
        worst += [check_zbc(S, p, 1) for p in FIRST_PATHS[:3]]
        worst += [check_book(S, p, 1) for p in FIRST_PATHS[:2]]
        worst += [check_curve(S, 7, 0, 1025), check_zbc(S, 7, 1, 1025)]
        print(f"{tag}: worst |gpu - f64| / pair_bound {max(worst):.3g}")
    finally:
        S.close()


# ---------------------------------------------------------------- aggregate
def second_bound(x, bx, y=None, by=None):
    """bound of sum x^2 (or sum x y) from per-summand bounds bx (by)"""
    if y is None:
        return (2 * np.abs(x) * bx + bx * bx).sum()
    return (np.abs(x) * by + np.abs(y) * bx + bx * by).sum()


def aggregate_line(what, got, ref, bound, sd, n, mode, a):
    se30 = sd / np.sqrt(2.0 ** 30)
    rel = np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)
    ratio = np.abs(got - ref) / n / np.maximum(se30, 1e-300)
    k = int(np.argmax(ratio))
    print(f"AGGREGATE mode {mode} a {a} {what}: worst |gpu - f64| / f64 {rel.max():.3g}, worst ratio of the mean's gap "
          f"to the 2^30-path standard error {ratio[k]:.3g} (entry {k})")
    assert (np.abs(got - ref) <= bound).all(), (what, float((np.abs(got - ref) / bound).max()))


@pytest.mark.parametrize("a", [1.0, 0.01])
def test_aggregate_bias(hw, engine, a):
    """2^18 pairs: every moment of the curve, ZBC and (a = 1) pathwise estimators against the f64 sums, relative to
    them, and the gap of each mean as a ratio to the standard error at 2^30 paths.  Bound: the summed per-pair bounds.
    Nobody has measured the MUFU bias of these kernels before: the printed figures are the record."""
    S = Setup(hw, engine, dict(a=a), table=(a != 1.0))
    try:
        n = 1 << 18
        F = S.F
        if refused(hw, engine, F):
            with pytest.raises(hw.HW1FError, match="decomposed mode is accurate only"):
                S.eng.bond_curve_moments(S.hw.Rng(SEED + 1, n), dev(2 * F.n_mat).data_ptr())
            return
        # curve: sum p0 and sum p0^2 at every save point
        m = dev(2 * F.n_mat)
        S.eng.bond_curve_moments(S.hw.Rng(SEED + 1, n), m.data_ptr())
        got = read(S, m)
        nm = F.n_mat
        ref, refq, b1, b2 = (np.zeros(nm - 1) for _ in range(4))
        steps = np.arange(1, nm) * F.stride
        sdI = np.array([F.sd_I(k * F.dt) for k in steps])
        for c in range(0, n, 1 << 15):
            st = F.states(SEED + 1, 1 << 15, steps, c, 0, drift=S.drift)
            p0 = np.exp(-st[:, :, 2]) + np.exp(-st[:, :, 3])
            bp = pair_bound(p0, rel_bound(steps, np.maximum(np.abs(st[:, :, 2]), np.abs(st[:, :, 3])), sdI))
            ref += p0.sum(0)
            refq += (p0 * p0).sum(0)
            b1 += bp.sum(0)
            b2 += (2 * p0 * bp + bp * bp).sum(0)
        sd = np.sqrt(np.maximum(refq / n - (ref / n) ** 2, 0.0))
        aggregate_line("curve sum p0", got[1:nm], ref, b1, sd, n, engine.mode, a)
        aggregate_line("curve sum p0^2", got[nm + 1:], refq, b2, sd, n, engine.mode, a)
        # ZBC: the five per-twin moments of hw1f_zbc_cv_moments
        nz = max(1, F.n_steps // 2)
        S1, z, rel = zbc_ref(S, 0, 1, n, nz)
        m = dev(5)
        S.eng.zbc_cv_moments(S.hw.Rng(SEED, n).seek(1), S.P, S.f, m.data_ptr(), S1=S1, S2=F.T_final, n_steps_S1=nz)
        got = read(S, m)
        x, y = z["x"], z["y"]
        bx, by = rel[:, None] * (x + y), rel[:, None] * y
        ref = np.array([x.sum(), y.sum(), (x * x).sum(), (y * y).sum(), (x * y).sum()])
        bound = np.array([bx.sum(), by.sum(), second_bound(x, bx), second_bound(y, by), second_bound(x, bx, y, by)])
        sd = np.array([x.std(), y.std(), (x * x).std(), (y * y).std(), (x * y).std()]) * np.sqrt(2.0)
        aggregate_line("zbc X, Y, X^2, Y^2, XY", got, ref, bound, sd, n, engine.mode, a)
        # pathwise: sum v, sum v^2 over the +G paths
        if S.exact:
            m = dev(2)
            S.eng.vega_pathwise_moments(S.hw.Rng(SEED, n).seek(1), S.P, S.f, m.data_ptr(), S1=S1, S2=F.T_final,
                                        n_steps_S1=nz)
            got = read(S, m)
            pw = F.pathwise(SEED, n, S.P, S.f, nz, S1=S1, S2=F.T_final, offset=1)
            zz, v = pw["zbc"], pw["v"][:, 0]
            r = rel_bound(nz, zz["I_abs"][:, 0], F.sd_I(S1), r_abs=zz["r_abs"][:, 0], B=zz["B"], sd_r=F.sd_r(S1))
            kink = np.abs(zz["P"][:, 0] - Oracle.K_DEFAULT) <= r * zz["P"][:, 0]
            bv = (pair_bound(pw["term1"][:, 0], r) + pair_bound(pw["term2"][:, 0], r, zz["y"][:, 0] * np.abs(pw["J"][:, 0]))
                  + np.where(kink, np.abs(pw["term1"][:, 0]), 0.0))
            aggregate_line("pathwise sum v, sum v^2", got, np.array([v.sum(), (v * v).sum()]),
                           np.array([bv.sum(), second_bound(v, bv)]) + 1e-12, np.array([v.std(), (v * v).std()]),
                           n, engine.mode, a)
    finally:
        S.close()
