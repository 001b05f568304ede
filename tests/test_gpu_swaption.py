"""European swaptions on the GPU (hw1f_swaptions*): a book of coupon-bond options in one simulation pass, in both
arithmetic modes, against the CPU oracle, the cap strip, Jamshidian's closed form, payer-receiver parity and its own
standard errors; the split form, every rejected argument, the edges of the schedule and model space, and runs whose
blocks stride over several chunks."""
import numpy as np
import pytest

import swaption_oracle
from cap_closed_form import continuous_theta, interp_mkt
from swaption_closed_form import book_closed_form, flows_of, forward_swap, par_rate
from swaption_oracle import moment_bound

pytestmark = pytest.mark.gpu

N = 1 << 13
SEED = 4321


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


def merge(*books):
    """one book from several (swaptions, flows) pairs, ordered by exercise date (stable)"""
    sws, fls, off = [], [], 0
    for sw, fl in books:
        sw = sw.copy()
        sw["first_flow"] += off
        off += len(fl)
        sws.append(sw)
        fls.append(fl)
    sw = np.concatenate(sws)
    return sw[np.argsort(sw["T_exercise"], kind="stable")], np.concatenate(fls)


def mixed_book(hw, P, T_final=10.0):
    """expiries 1-9 with several tenors each (shared exercise steps), odd exercise steps 255, 437 and 611, annual and
    semi-annual flows, payer and receiver options alternating, strikes at and around the money"""
    books = []
    for freq, Te, ten in (
            (1, [1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 2.55, 4.37], [1, 9, 1, 8, 1, 7, 1, 6, 1, 5, 1, 4, 1, 3,
                                                                                1, 2, 1, 3, 5]),
            (2, [1, 1, 3, 3, 5, 5, 7, 7, 9, 6.11], [2, 9, 2, 7, 2, 5, 2, 3, 1, 2])):
        Te, ten = np.array(Te, np.float64), np.array(ten, np.float64)
        shift = 0.005 * ((np.arange(len(Te)) % 3) - 1)
        kappa = [par_rate(P, T_final, t, n, freq) + s for t, n, s in zip(Te, ten, shift)]
        kinds = ["payer" if (k + freq) % 2 else "receiver" for k in range(len(Te))]
        books.append(hw.swaption_schedule(Te, ten, kappa, freq=freq, notional=100.0, kind=kinds))
    return merge(*books)


def all_moments(res):
    return np.vstack([res["mom"], np.asarray(res["book"]["mom"])[None, :]])


def check(got, ref, rel=3e-6, what=""):
    mom = all_moments(got)
    gap, bound = np.abs(mom - ref), moment_bound(ref, rel=rel)
    print(f"{what}: worst moment gap / bound {(gap / bound).max():.3g}")
    assert np.isfinite(mom).all()
    assert (gap <= bound).all(), (what, np.unravel_index((gap / bound).argmax(), gap.shape), (gap / bound).max())


# hw1f_swaption / hw1f_cash_flow (include/hw1f.h)
SW_DTYPE = np.dtype([("T_exercise", "f4"), ("K", "f4"), ("N", "f4"), ("kind", "i4"), ("n_steps_exercise", "i4"),
                     ("first_flow", "i4"), ("n_flows", "i4"), ("reserved", "i4")])
FLOW_DTYPE = np.dtype([("T", "f4"), ("c", "f4")])


def one(Te, flows, K, N_, kind="payer", step=-1):
    """one option on the flows [(T, c), ...]"""
    sw = np.array([(Te, K, N_, 0 if kind == "payer" else 1, step, 0, len(flows), 0)], SW_DTYPE)
    return sw, np.array(flows, FLOW_DTYPE).reshape(len(flows))


# ---------------------------------------------------------------- 1. against the oracle
@pytest.mark.parametrize("offset", [0, 499])
def test_book_moments_vs_oracle(engine, hw, oracle, curve, offset):
    sw, fl = mixed_book(hw, curve["P"])
    assert len(np.unique(sw["T_exercise"])) < len(sw) and (sw["kind"] == 0).any() and (sw["kind"] == 1).any()
    rng = hw.Rng(SEED + 99, N).seek(offset)
    got = engine.swaptions(rng, sw, fl, curve["P"], curve["f"])
    assert rng.tell() == offset + 900
    ref = swaption_oracle.swaption_moments(oracle, SEED + 99, N, sw, fl, curve["P"], curve["f"], offset=offset)
    check(got, ref, what=f"mixed book offset {offset}")


# ---------------------------------------------------------------- 2. one flow = one caplet
@pytest.mark.parametrize("kind", ["payer", "receiver"])
def test_one_flow_is_one_caplet(engine, hw, curve, kind):
    K, N_ = engine.K_DEFAULT, 1.75
    sw, fl = one(5.0, [(10.0, 1.0)], K, N_, kind=kind)
    caps = np.array([(5.0, 10.0, K, N_, -1, 0)], [("T_reset", "f4"), ("T_pay", "f4"), ("K", "f4"), ("N", "f4"),
                                                   ("n_steps_reset", "i4"), ("reserved", "i4")])
    r1, r2 = hw.Rng(SEED + 7, N).seek(3), hw.Rng(SEED + 7, N).seek(3)
    s = engine.swaptions(r1, sw, fl, curve["P"], curve["f"])
    c = engine.cap_floor(r2, caps, curve["P"], curve["f"], kind="cap" if kind == "payer" else "floor")
    assert r1.tell() == r2.tell() == 503
    a, b = all_moments(s), np.vstack([c["mom"], np.asarray(c["strip"]["mom"])[None, :]])
    print(f"{kind}: one-flow swaption bit-identical to the caplet: {np.array_equal(a, b)}, "
          f"worst relative gap {np.max(np.abs(a - b) / np.abs(b)):.3g}")
    assert (np.abs(a - b) <= 1e-6 * np.abs(b)).all(), (a, b)
    assert s["control_mean"][0] == c["control_mean"][0]


# ---------------------------------------------------------------- 3, 4. Jamshidian and payer-receiver parity
@pytest.fixture(scope="module")
def cf_setup(engine, hw):
    eng = hw.Engine(device=0, params=hw.default_params(**continuous_theta()))
    eng.set_mode(engine.mode)
    c = eng.bond_curve(hw.Rng(20252, 1 << 21))
    yield eng, c
    eng.close()


def grid_book(hw, P, T_final, kinds=("payer", "receiver")):
    """3 x 3 expiry x tenor grid (semi-annual), ATM and +-100 bp, each as every kind in `kinds`"""
    Te, ten, kap, kd = [], [], [], []
    for e in (1.0, 3.0, 5.0):
        for t in (1.0, 2.0, 5.0):
            atm = par_rate(P, T_final, e, t, 2)
            for dk in (-0.01, 0.0, 0.01):
                for k in kinds:
                    Te.append(e); ten.append(t); kap.append(atm + dk); kd.append(k)
    return hw.swaption_schedule(Te, ten, kap, freq=2, notional=100.0, kind=kd)


def test_grid_vs_jamshidian_and_parity(cf_setup, hw):
    eng, c = cf_setup
    P, f, P_se = c["P"], c["f"], c["P_se"]
    p = eng.params
    sw, fl = grid_book(hw, P, p.T_final)
    assert len(sw) == 54
    g = eng.swaptions(hw.Rng(41, 1 << 20), sw, fl, P, f)
    cf = np.array(book_closed_form(sw, fl, P, f, p.a, p.sigma, p.T_final))
    up = np.array(book_closed_form(sw, fl, P + P_se, f, p.a, p.sigma, p.T_final))
    dn = np.array(book_closed_form(sw, fl, P - P_se, f, p.a, p.sigma, p.T_final))
    allow = np.abs(up - dn)
    dev = np.abs(g["price_cv"] - cf)
    print(f"worst |MC - Jamshidian| / se_cv {np.max(dev / g['se_cv']):.3g}; "
          f"worst |MC - Jamshidian| / (4 se_cv + allowance) {np.max(dev / (4 * g['se_cv'] + allow)):.3g}")
    assert (dev <= 4 * g["se_cv"] + allow).all(), (dev / g["se_cv"], allow)
    assert abs(g["book"]["price_cv"] - cf.sum()) <= 4 * g["book"]["se_cv"] + allow.sum(), (g["book"], cf.sum())
    assert g["book"]["price_raw"] == pytest.approx(g["price_raw"].sum(), rel=1e-6)
    # payer - receiver = N (K P0(T_e) - sum_j c_j P0(T_j)), in one call
    n_mat = len(P)
    for i in range(0, len(sw), 2):
        assert sw["kind"][i] == 0 and sw["kind"][i + 1] == 1 and sw["first_flow"][i] != sw["first_flow"][i + 1]
        Ts, cs = flows_of(sw[i], fl)
        Te, K, N_ = float(sw["T_exercise"][i]), float(sw["K"][i]), float(sw["N"][i])
        diff = g["price_cv"][i] - g["price_cv"][i + 1]
        se = np.hypot(g["se_cv"][i], g["se_cv"][i + 1])
        fwd = forward_swap(P, p.T_final, Te, Ts, cs, K, N_)
        band = abs(forward_swap(P + P_se, p.T_final, Te, Ts, cs, K, N_) - forward_swap(P - P_se, p.T_final, Te, Ts, cs, K, N_))
        assert abs(diff - fwd) <= 4 * se + band, (i, diff, fwd, se, band)
        cm = N_ * sum(cj * interp_mkt(P, T, p.T_final, n_mat) for T, cj in zip(Ts, cs))
        assert g["control_mean"][i] == pytest.approx(cm, rel=1e-12)


# ---------------------------------------------------------------- 5. standard errors
def test_standard_errors_are_honest(engine, hw, curve):
    sw, fl = mixed_book(hw, curve["P"])
    seeds = [700003 + 7919 * k for k in range(40)]
    runs = [engine.swaptions(hw.Rng(s, 1 << 16), sw, fl, curve["P"], curve["f"]) for s in seeds]
    for est, se in (("price_cv", "se_cv"), ("price_raw", "se_raw")):
        book = np.array([r["book"][est] for r in runs])
        ratio = np.mean([r["book"][se] for r in runs]) / book.std(ddof=1)
        assert 0.75 < ratio < 1.25, (est, ratio)
        x = np.array([r[est] for r in runs])
        rc = np.array([r[se] for r in runs]).mean(axis=0) / x.std(axis=0, ddof=1)
        print(f"{est}: book se / spread {ratio:.3f}, per option median {np.median(rc):.3f} [{rc.min():.3f}, {rc.max():.3f}]")
        assert 0.75 < np.median(rc) < 1.25, (est, np.median(rc))
        assert rc.min() > 0.55 and rc.max() < 1.6, (est, rc.min(), rc.max())


# ---------------------------------------------------------------- 6. split form
def test_split_form_and_reproducibility(engine, hw, curve):
    import torch
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    nq = 5 * (len(sw) + 1)
    full = torch.zeros(nq, dtype=torch.float64, device="cuda")
    a_part, b_part = torch.zeros_like(full), torch.zeros_like(full)
    a = 3 * 1024 + 17
    torch.cuda.synchronize()
    rng = hw.Rng(SEED + 5, N).seek(3)
    engine.swaptions_moments(rng, sw, fl, P, f, full.data_ptr())
    assert rng.tell() == 3 + 900
    engine.swaptions_moments(hw.Rng(SEED + 5, a).seek(3), sw, fl, P, f, a_part.data_ptr())
    engine.swaptions_moments(hw.Rng(SEED + 5, N - a, first_path=a).seek(3), sw, fl, P, f, b_part.data_ptr())
    engine.synchronize()
    f_, s_ = full.cpu().numpy(), (a_part + b_part).cpu().numpy()
    assert np.allclose(f_, s_, rtol=2e-6, atol=0), np.abs(f_ / s_ - 1).max()
    fin = engine.swaptions_finish(full.data_ptr(), N, sw, fl, P)
    one_call = engine.swaptions(hw.Rng(SEED + 5, N).seek(3), sw, fl, P, f)
    for k in ("price_cv", "se_cv", "price_raw", "se_raw", "beta", "corr", "control_mean", "mom"):
        assert np.array_equal(fin[k], one_call[k]), k
    assert fin["book"] == one_call["book"]
    again = engine.swaptions(hw.Rng(SEED + 5, N).seek(3), sw, fl, P, f)
    assert np.array_equal(again["mom"], one_call["mom"]) and again["book"] == one_call["book"]


# ---------------------------------------------------------------- 7. rejected arguments
def rejected_cases(engine, hw):
    Tf, n_steps = float(engine.params.T_final), engine.n_steps
    good = one(1.0, [(1.5, 0.02), (2.0, 1.02)], 1.0, 1.0)

    def edit(book, **kw):
        sw, fl = book[0].copy(), book[1].copy()
        for k, v in kw.items():
            if k in sw.dtype.names:
                sw[k] = v
            else:
                fl[k[:-1]][int(k[-1])] = v          # "T0" / "c1": flow 0's T, flow 1's c
        return sw, fl

    sw2, fl2 = merge(one(0.5, [(1.0, 1.0)], 1.0, 1.0), one(0.25, [(1.0, 1.0)], 1.0, 1.0))
    many = np.float32(1.0 + 8.5 * np.arange(1, 1026) / 1025.0)
    big = one(1.0, [(float(t), 0.01) for t in many], 1.0, 1.0)
    shared = (np.concatenate([big[0], big[0]]), big[1])                  # 2 x 1025 rows of one flow table
    huge = one(0.5, [(float(t), 0.01) for t in np.float32(0.5 + 9.5 * np.arange(1, 2050) / 2049.0)], 1.0, 1.0)
    return [
        ("kind", edit(good, kind=2)),
        ("kind negative", edit(good, kind=-1)),
        ("n_swaptions 0", (good[0][:0], good[1])),
        ("n_swaptions 101", (np.repeat(good[0], 101), good[1])),
        ("no flows", (good[0], good[1][:0])),
        ("sum of n_flows 2050", shared),
        ("one option of 2049 flows", huge),
        ("option n_flows 0", edit(good, n_flows=0)),
        ("flow range beyond flows", edit(good, first_flow=1)),
        ("first_flow negative", edit(good, first_flow=-1)),
        ("flow dates not increasing", edit(good, T1=1.5)),
        ("first flow at T_exercise", edit(good, T0=1.0)),
        ("last flow beyond T_final", edit(good, T1=Tf + 0.5)),
        ("flow date nan", edit(good, T0=np.nan)),
        ("c = 0", edit(good, c0=0.0)),
        ("c < 0 (forward start)", edit(good, c0=-1.0)),
        ("c = inf", edit(good, c1=np.inf)),
        ("K = 0", edit(good, K=0.0)),
        ("K = nan", edit(good, K=np.nan)),
        ("N < 0", edit(good, N=-1.0)),
        ("N = inf", edit(good, N=np.inf)),
        ("T_exercise off the grid", edit(good, T_exercise=1.0037)),
        ("T_exercise 0", edit(good, T_exercise=0.0)),
        ("step 0", edit(good, n_steps_exercise=0)),
        ("step beyond n_steps", edit(good, n_steps_exercise=n_steps + 1)),
        ("decreasing steps", (sw2[::-1].copy(), fl2)),
    ]


def test_rejected_arguments(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    for name, (sw, fl) in rejected_cases(engine, hw):
        rng = hw.Rng(SEED, N).seek(7)
        before = engine.launch_count
        with pytest.raises(hw.HW1FError) as ei:
            engine.swaptions(rng, sw, fl, P, f)
        assert ei.value.status == hw._ffi.ERR_INVALID, name
        assert len(str(ei.value).split(":", 1)[1].strip()) > 10, (name, str(ei.value))
        with pytest.raises(hw.HW1FError) as ei:
            engine.swaptions_moments(rng, sw, fl, P, f, 0)
        assert ei.value.status == hw._ffi.ERR_INVALID, name
        assert engine.launch_count == before, name
        assert rng.tell() == 7, name


# ---------------------------------------------------------------- 8. edges
def test_never_paying_option(engine, hw, oracle, curve):
    P, f = curve["P"], curve["f"]
    sw, fl = merge(one(2.0, [(3.0, 0.03), (4.0, 1.03)], 0.01, 100.0, kind="payer"),       # Bnd >> K: the put never pays
                   one(2.0, [(3.0, 0.03), (4.0, 1.03)], 5.0, 100.0, kind="receiver"),     # Bnd << K: the call never pays
                   one(3.0, [(4.0, 0.03), (5.0, 1.03)], 1.0, 100.0, kind="payer"))
    got = engine.swaptions(hw.Rng(SEED + 3, N).seek(2), sw, fl, P, f)
    for k in ("price_raw", "price_cv", "se_raw", "se_cv", "beta", "corr", "control_mean"):
        assert np.isfinite(got[k]).all() and np.isfinite(got["book"][k]), k
        if k != "control_mean":
            assert (got[k][:2] == 0.0).all(), k                     # X == 0 on every path: no 0/0
    assert (got["mom"][:2][:, [0, 2, 4]] == 0).all()
    assert got["price_raw"][2] > 0
    ref = swaption_oracle.swaption_moments(oracle, SEED + 3, N, sw, fl, P, f, offset=2)
    check(got, ref, what="never paying")


def test_exercise_at_first_and_last_step(engine, hw, oracle, curve):
    P, f = curve["P"], curve["f"]
    ns, Tf = engine.n_steps, float(engine.params.T_final)
    dt = Tf / ns
    first = one(dt, [(0.5, 0.02), (1.0, 1.02)], 1.0, 10.0, kind="receiver", step=1)
    # the last step: T_exercise a hair below T_final (the step is given), its only flow at T_final
    last = one(Tf - dt, [(Tf, 1.0)], 0.9997, 10.0, kind="payer", step=ns)       # about at the money
    sw, fl = merge(first, last)
    for off in (0, 1):
        rng = hw.Rng(SEED + 11, N).seek(off)
        got = engine.swaptions(rng, sw, fl, P, f)
        assert rng.tell() == off + ns
        ref = swaption_oracle.swaption_moments(oracle, SEED + 11, N, sw, fl, P, f, offset=off)
        # one step from r0: every path sits at almost the same r, so the MUFU-vs-libm difference of the payoff does not
        # average out (test_zbc_moments_vs_oracle's allowance for 1-2 steps)
        check(got, ref, rel=2e-4, what=f"first and last step, offset {off}")


def hundred_on_longest(hw, P, ns, Tf):
    steps = np.linspace(3, ns - 3, 100).round().astype(int)
    dt = Tf / ns
    nf = np.full(100, 20)
    nf[:48] = 21
    assert nf.sum() == 2048
    books = []
    for k, m, i in zip(steps, nf, range(100)):
        Te = float(np.float32(k * dt))
        T = np.minimum(np.float32(Te + (Tf - Te) * np.arange(1, m + 1) / m), np.float32(Tf))
        c = np.full(m, 0.03 / m)
        c[-1] += 1.0
        books.append(one(Te, list(zip(T.tolist(), c.tolist())), 1.0, 1.0, kind="payer" if i % 2 else "receiver",
                         step=int(k)))
    sw, fl = merge(*books)
    assert len(sw) == 100 and len(fl) == 2048 and len(np.unique(steps)) == 100
    assert all((np.diff(fl["T"][s:s + n]) > 0).all() for s, n in zip(sw["first_flow"], sw["n_flows"]))
    return sw, fl


def test_hundred_swaptions_2048_flows_on_the_longest_grid(engine, hw):
    """HW1F_MAX_SWAPTIONS and HW1F_MAX_SWAPTION_FLOWS on 8184 steps: the largest shared-memory footprint (reference
    order: ~108 KB).  It must price; a refusal would be HW1F_ERR_UNSUPPORTED, never a wrong number."""
    from oracle_lib import Oracle
    over = dict(n_steps=8184, n_mat=1024)
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(engine.mode)
    try:
        n, ns, Tf = 1 << 10, eng.n_steps, float(eng.params.T_final)
        c = eng.bond_curve(hw.Rng(31339, 1 << 12))
        sw, fl = hundred_on_longest(hw, c["P"], ns, Tf)
        got = eng.swaptions(hw.Rng(8, n).seek(1), sw, fl, c["P"], c["f"])
        ref = swaption_oracle.swaption_moments(o, 8, n, sw, fl, c["P"], c["f"], offset=1)
        check(got, ref, rel=5e-6, what="100 swaptions, 2048 flows")
    finally:
        eng.close()


def test_smallest_model(engine, hw):
    from oracle_lib import Oracle
    over = dict(n_steps=2, n_mat=3, T_final=0.5)
    o = Oracle(**over)
    eng = hw.Engine(device=0, params=hw.default_params(**over))
    eng.set_mode(engine.mode)
    try:
        n = 1 << 12
        c = eng.bond_curve(hw.Rng(31340, n))
        K = float(c["P"][2] / c["P"][1] * 1.0001 + 0.0001)
        sw, fl = merge(one(0.25, [(0.375, 0.0001), (0.5, 1.0)], K, 1.0, kind="payer"),
                       one(0.25, [(0.5, 1.0)], K, 1.0, kind="receiver"))
        for off in (0, 1):
            got = eng.swaptions(hw.Rng(9, n).seek(off), sw, fl, c["P"], c["f"])
            ref = swaption_oracle.swaption_moments(o, 9, n, sw, fl, c["P"], c["f"], offset=off)
            check(got, ref, rel=2e-4, what=f"2 x 3 model, offset {off}")    # one step: see test_exercise_at_first_and_last_step
    finally:
        eng.close()


def test_new_entry_points_as_first_call_of_a_fresh_engine(engine, hw, curve):
    import torch
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    want = engine.swaptions(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f)
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        got = e.swaptions(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f)
    finally:
        e.close()
    assert np.array_equal(got["mom"], want["mom"]) and got["book"] == want["book"]
    mom = torch.zeros(5 * (len(sw) + 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        e.swaptions_moments(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f, mom.data_ptr())
        e.synchronize()
        fin = e.swaptions_finish(mom.data_ptr(), N + 5, sw, fl, P)
    finally:
        e.close()
    assert np.array_equal(fin["mom"], want["mom"]) and fin["book"] == want["book"]


# ---------------------------------------------------------------- 9. blocks that stride over several chunks
KCHUNK = 1024
MODEL = dict(n_steps=40, n_mat=11, T_final=0.4)   # dt 0.01
FIRST = 300
GS_SEED = 4243


def chunk_count(first, n):
    return (first + n - 1) // KCHUNK - first // KCHUNK + 1


@pytest.fixture(scope="module")
def geom():
    import torch
    grid = 32 * torch.cuda.get_device_properties(0).multi_processor_count      # prepare_launch's grid cap
    n = (2 * grid + 37) * KCHUNK + 5
    n_chunks = chunk_count(FIRST, n)
    assert 2 * grid < n_chunks < 3 * grid, (grid, n_chunks)
    b1 = (grid - 1) * KCHUNK
    b2 = (2 * grid - 3) * KCHUNK + 517
    shards = [(FIRST, b1 - FIRST), (b1, b2 - b1), (b2, FIRST + n - b2)]
    assert all(chunk_count(f_, c) <= grid for f_, c in shards)
    return dict(grid=grid, n=n, shards=shards)


def short_book(hw, P):
    """exercise steps 1, 4, 8, 8, 17, 19, 24, 31, 37 (gaps 1, 3, 4, 0, 9, 2, 5, 7, 6), flows every 0.01 to 0.05"""
    steps = np.array([1, 4, 8, 8, 17, 19, 24, 31, 37])
    n_fl = np.array([3, 2, 5, 1, 4, 3, 2, 1, 3])
    books = []
    for i, (k, m) in enumerate(zip(steps, n_fl)):
        Te = float(np.float32(k * 0.01))
        T = np.float32(Te + 0.01 * np.arange(1, m + 1))
        c = np.full(m, 0.002)
        c[-1] += 1.0
        K = float(sum(cj * interp_mkt(P, t, 0.4, 11) for t, cj in zip(T, c)) / interp_mkt(P, Te, 0.4, 11))
        books.append(one(Te, list(zip(T.tolist(), c.tolist())), K, 50.0, kind="payer" if i % 2 else "receiver",
                         step=int(k)))
    return merge(*books)


@pytest.fixture(scope="module")
def gs_ref(geom, hw):
    from oracle_lib import Oracle
    o = Oracle(**MODEL)
    n = geom["n"]
    s, _ = o.bond_curve_sums(GS_SEED, n, first_path=FIRST)
    P, f = o.curve_finalize(s, n)
    sw, fl = short_book(hw, P)
    return dict(P=P, f=f, sw=sw, fl=fl,
                mom=swaption_oracle.swaption_moments(o, GS_SEED + 1, n, sw, fl, P, f, first_path=FIRST, offset=1))


@pytest.fixture(scope="module")
def short(engine, hw):
    e = hw.Engine(device=0, params=hw.default_params(**MODEL))
    e.set_mode(engine.mode)
    yield e
    e.close()


def test_grid_stride_vs_oracle_and_shards(short, hw, geom, gs_ref):
    import torch
    n, P, f, sw, fl = geom["n"], gs_ref["P"], gs_ref["f"], gs_ref["sw"], gs_ref["fl"]
    rng = hw.Rng(GS_SEED + 1, n, first_path=FIRST).seek(1)      # odd offset: every chunk starts on a cached cos half
    got = short.swaptions(rng, sw, fl, P, f)
    assert rng.tell() == 1 + 37
    check(got, gs_ref["mom"], what="grid stride vs oracle")
    # full range == sum of one-pass shards (test_gpu_grid_stride's FLOAT_TREES bound: a missing or doubled chunk moves
    # a sum by ~1e-4)
    nq = 5 * (len(sw) + 1)
    full = torch.zeros(nq, dtype=torch.float64, device="cuda")
    acc, part = torch.zeros_like(full), torch.zeros_like(full)
    torch.cuda.synchronize()
    short.swaptions_moments(hw.Rng(GS_SEED + 5, n, first_path=FIRST).seek(1), sw, fl, P, f, full.data_ptr())
    short.synchronize()
    for first, cnt in geom["shards"]:
        short.swaptions_moments(hw.Rng(GS_SEED + 5, cnt, first_path=first).seek(1), sw, fl, P, f, part.data_ptr())
        short.synchronize()
        acc += part
        torch.cuda.synchronize()          # the next launch overwrites `part`
    a, b = full.cpu().numpy(), acc.cpu().numpy()
    assert np.isfinite(a).all()
    nz = a != 0
    rel = np.abs(a[nz] - b[nz]) / np.abs(a[nz])
    print(f"worst relative gap full vs shards {rel.max():.3g}")
    assert (rel <= 1e-9).all() and (b[~nz] == 0).all(), rel.max()
