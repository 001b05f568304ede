"""Vega of swaption books and cap strips on the GPU (hw1f_swaptions_vega*): the book priced at sigma, sigma - eps and
sigma + eps on one set of normals, in both arithmetic modes.  Checked: the base block against hw1f_swaptions bit for
bit, the vega block against the CPU oracle, that fd_theta_a1 is not read and hw1f_vega_fd is not disturbed, Jamshidian
and the caplet closed form, honest standard errors, the split form, every rejected argument and the edges."""
import ctypes as C

import numpy as np
import pytest

import swaption_vega_oracle as svo
from cap_closed_form import atm_rate, continuous_theta, strip_closed_form
from swaption_closed_form import book_closed_form, par_rate
from swaption_oracle import moment_bound
from test_gpu_swaption import hundred_on_longest, merge, mixed_book, one, rejected_cases, short_book

pytestmark = pytest.mark.gpu

N = 1 << 13
SEED = 5821
EPS = 1e-3
VEGA_KEYS = ("price_minus", "se_minus", "price_plus", "se_plus", "vega", "vega_se", "vega_mom")
BASE_KEYS = ("price_cv", "se_cv", "price_raw", "se_raw", "beta", "corr", "control_mean", "mom")


@pytest.fixture(scope="module")
def curve(engine, hw):
    return engine.bond_curve(hw.Rng(SEED, N))


def engine_like(engine, hw, **over):
    e = hw.Engine(device=0, params=hw.default_params(**over))
    e.set_mode(engine.mode)
    return e


def blocks(res):
    """(base[n + 1, 5], vega[n + 1, 6]) of a swaptions_vega result"""
    base = np.vstack([res["mom"], np.asarray(res["book"]["mom"])[None, :]])
    vega = np.vstack([res["vega_mom"], np.asarray(res["book"]["vega_mom"])[None, :]])
    return base, vega


def check_vs_oracle(got, ref, aux, n, rel=3e-6, what=""):
    base, vega = blocks(got)
    rb, rv = svo.split(ref, n)
    gb, bb = np.abs(base - rb), moment_bound(rb, rel=rel)
    gv, bv = np.abs(vega - rv), svo.vega_bound(rv, aux, rel=rel)
    print(f"{what}: worst gap / bound base {(gb / bb).max():.3g}, vega block {(gv / bv).max():.3g}")
    assert np.isfinite(base).all() and np.isfinite(vega).all()
    assert (gb <= bb).all(), (what, np.unravel_index((gb / bb).argmax(), gb.shape), (gb / bb).max())
    assert (gv <= bv).all(), (what, np.unravel_index((gv / bv).argmax(), gv.shape), (gv / bv).max())


def same_result(a, b, book="book"):
    for k in BASE_KEYS + VEGA_KEYS:
        assert np.array_equal(a[k], b[k]), k
    assert a[book] == b[book]


# ---------------------------------------------------------------- 1. the base block is hw1f_swaptions
def test_base_block_is_swaptions_bit_for_bit(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    r1, r2 = hw.Rng(SEED + 1, N).seek(5), hw.Rng(SEED + 1, N).seek(5)
    s = engine.swaptions(r1, sw, fl, P, f)
    v = engine.swaptions_vega(r2, sw, fl, P, f, eps=EPS)
    assert r1.tell() == r2.tell() == 905
    for k in BASE_KEYS:
        assert np.array_equal(s[k], v[k]), k
    assert all(v["book"][k] == s["book"][k] for k in s["book"])
    assert v["sim_ms"] > 0


# ---------------------------------------------------------------- 2. against the oracle
@pytest.mark.parametrize("offset", [0, 499])
def test_vega_moments_vs_oracle(engine, hw, oracle, curve, offset):
    """default params: theta_a1 (0.019) != fd_theta_a1 (0.014), and the mixed book exercises up to year 9"""
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    assert sw["T_exercise"].max() > oracle.p.theta_break
    rng = hw.Rng(SEED + 99, N).seek(offset)
    got = engine.swaptions_vega(rng, sw, fl, P, f, eps=EPS)
    assert rng.tell() == offset + 900
    ref, aux = svo.vega_moments(oracle, SEED + 99, N, sw, fl, P, f, EPS, offset=offset)
    check_vs_oracle(got, ref, aux, len(sw), what=f"mixed book offset {offset}")


# ---------------------------------------------------------------- 3, 4. fd_theta_a1 and hw1f_vega_fd
def test_fd_theta_a1_is_not_read(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    want = engine.swaptions_vega(hw.Rng(SEED + 2, N).seek(1), sw, fl, P, f, eps=EPS)
    e = engine_like(engine, hw, fd_theta_a1=0.5)
    try:
        got = e.swaptions_vega(hw.Rng(SEED + 2, N).seek(1), sw, fl, P, f, eps=EPS)
    finally:
        e.close()
    same_result(got, want)


def test_vega_fd_is_untouched(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)

    def fd(eps):
        return engine.vega_fd(hw.Rng(SEED + 3, N), P, f, eps=eps)
    before = fd(EPS)
    engine.swaptions_vega(hw.Rng(SEED + 4, N), sw, fl, P, f, eps=EPS)
    mid = fd(EPS)
    engine.swaptions_vega(hw.Rng(SEED + 4, N), sw, fl, P, f, eps=2e-3)
    fd(5e-4)
    engine.swaptions_vega(hw.Rng(SEED + 4, N), sw, fl, P, f, eps=5e-4)
    after = fd(EPS)
    for r in (mid, after):
        for k in ("price_minus", "price_plus", "vega_fd", "n_steps_S1"):     # everything but the timings
            assert r[k] == before[k], k


# ---------------------------------------------------------------- 5. Jamshidian at sigma -/+ eps
@pytest.fixture(scope="module")
def cf_setup(engine, hw):
    eng = engine_like(engine, hw, **continuous_theta())
    c = eng.bond_curve(hw.Rng(20252, 1 << 21))
    yield eng, c
    eng.close()


def grid_book(hw, P, T_final):
    """the 54-option grid of test_gpu_swaption: expiries 1, 3, 5 x tenors 1, 2, 5, ATM and +-100 bp, payer and receiver"""
    Te, ten, kap, kd = [], [], [], []
    for e in (1.0, 3.0, 5.0):
        for t in (1.0, 2.0, 5.0):
            atm = par_rate(P, T_final, e, t, 2)
            for dk in (-0.01, 0.0, 0.01):
                for k in ("payer", "receiver"):
                    Te.append(e); ten.append(t); kap.append(atm + dk); kd.append(k)
    return hw.swaption_schedule(Te, ten, kap, freq=2, notional=100.0, kind=kd)


def bumped_sigmas(sigma, eps):
    e32 = float(np.float32(eps))
    return float(np.float32(sigma - e32)), float(np.float32(sigma + e32)), e32


def jamshidian_check(g, sw, fl, P, f, P_se, p, with_vega, what):
    sm, sp, e32 = bumped_sigmas(p.sigma, EPS)

    def cf(P_, s_):
        return np.array(book_closed_form(sw, fl, P_, f, p.a, s_, p.T_final))
    worst = 0.0
    for key, se, s_ in (("price_minus", "se_minus", sm), ("price_plus", "se_plus", sp)):
        want = cf(P, s_)
        allow = np.abs(cf(P + P_se, s_) - cf(P - P_se, s_))
        dev = np.abs(g[key] - want)
        worst = max(worst, np.max(dev / (4 * g[se] + allow)))
        assert (dev <= 4 * g[se] + allow).all(), (what, key, dev / g[se], allow)
    if with_vega:
        def vcf(P_):
            return (cf(P_, sp) - cf(P_, sm)) / (2 * e32)
        want = vcf(P)
        allow = np.abs(vcf(P + P_se) - vcf(P - P_se))
        dev = np.abs(g["vega"] - want)
        worst = max(worst, np.max(dev / (4 * g["vega_se"] + allow)))
        print(f"{what}: worst |vega - Jamshidian| / vega_se {np.max(dev / g['vega_se']):.3g}")
        assert (dev <= 4 * g["vega_se"] + allow).all(), (what, dev / g["vega_se"], allow)
        assert abs(g["book"]["vega"] - want.sum()) <= 4 * g["book"]["vega_se"] + allow.sum(), (g["book"], want.sum())
    print(f"{what}: worst |MC - Jamshidian| / (4 se + allowance) {worst:.3g}")


def test_grid_vega_vs_jamshidian(cf_setup, hw):
    eng, c = cf_setup
    P, f, P_se = c["P"], c["f"], c["P_se"]
    p = eng.params
    sw, fl = grid_book(hw, P, p.T_final)
    assert len(sw) == 54
    g = eng.swaptions_vega(hw.Rng(41, 1 << 20), sw, fl, P, f, eps=EPS)
    jamshidian_check(g, sw, fl, P, f, P_se, p, True, "54-option grid, continuous theta")
    assert (g["vega"] > 0).all()


def test_default_params_after_theta_break_vs_jamshidian(engine, hw):
    """expiries 6-8 years on the default model: a bumped model that read fd_theta_a1 would have theta lower by 0.005
    there, and its prices would miss the closed form on the (fixed) curve"""
    c = engine.bond_curve(hw.Rng(20253, 1 << 21))
    P, f, P_se = c["P"], c["f"], c["P_se"]
    p = engine.params
    Te = np.array([6.0, 6.0, 7.0, 7.0, 8.0, 8.0])
    ten = np.array([1.0, 2.0, 1.0, 2.0, 1.0, 2.0])
    kap = [par_rate(P, p.T_final, t, n, 2) for t, n in zip(Te, ten)]
    sw, fl = hw.swaption_schedule(Te, ten, kap, freq=2, notional=100.0, kind=["payer", "receiver"] * 3)
    g = engine.swaptions_vega(hw.Rng(43, 1 << 20), sw, fl, P, f, eps=EPS)
    jamshidian_check(g, sw, fl, P, f, P_se, p, False, "default params, expiries 6-8")


# ---------------------------------------------------------------- 6. caps
def caplets(hw, P, T_final, n=39, tau=0.25):
    resets = tau * np.arange(1, n + 1)
    pays = resets + tau
    return hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, T_final), notional=100.0)


@pytest.mark.parametrize("kind", ["cap", "floor"])
def test_cap_floor_vega_base_is_the_strip(engine, hw, curve, kind):
    P, f = curve["P"], curve["f"]
    cap = caplets(hw, P, float(engine.params.T_final), n=9, tau=1.0)
    r1, r2 = hw.Rng(SEED + 7, N).seek(3), hw.Rng(SEED + 7, N).seek(3)
    v = engine.cap_floor_vega(r1, cap, P, f, kind=kind, eps=EPS)
    c = engine.cap_floor(r2, cap, P, f, kind=kind)
    assert r1.tell() == r2.tell()
    a = np.vstack([v["mom"], np.asarray(v["strip"]["mom"])[None, :]])
    b = np.vstack([c["mom"], np.asarray(c["strip"]["mom"])[None, :]])
    assert np.array_equal(a, b), (a, b)
    assert np.array_equal(v["control_mean"], c["control_mean"])
    assert (v["vega"] > 0).all() and v["strip"]["vega"] > 0


def test_cap_vega_vs_closed_form(cf_setup, hw):
    eng, c = cf_setup
    P, f, P_se = c["P"], c["f"], c["P_se"]
    p = eng.params
    cap = caplets(hw, P, p.T_final)
    g = eng.cap_floor_vega(hw.Rng(45, 1 << 20), cap, P, f, kind="cap", eps=EPS)
    sm, sp, e32 = bumped_sigmas(p.sigma, EPS)

    def vcf(P_):
        return (strip_closed_form("cap", cap, P_, p.a, sp, p.T_final)[0] -
                strip_closed_form("cap", cap, P_, p.a, sm, p.T_final)[0]) / (2 * e32)
    want = vcf(P)
    allow = np.abs(vcf(P + P_se) - vcf(P - P_se))
    dev = np.abs(g["vega"] - want)
    print(f"39-caplet cap: worst |vega - closed form| / vega_se {np.max(dev / g['vega_se']):.3g}")
    assert (dev <= 4 * g["vega_se"] + allow).all(), (dev / g["vega_se"], allow)
    assert abs(g["strip"]["vega"] - want.sum()) <= 4 * g["strip"]["vega_se"] + allow.sum(), (g["strip"], want.sum())


# ---------------------------------------------------------------- 7. standard errors
def test_standard_errors_are_honest(engine, hw, curve):
    sw, fl = mixed_book(hw, curve["P"])
    seeds = [700003 + 7919 * k for k in range(40)]
    runs = [engine.swaptions_vega(hw.Rng(s, 1 << 16), sw, fl, curve["P"], curve["f"], eps=EPS) for s in seeds]
    for est, se in (("vega", "vega_se"), ("price_minus", "se_minus"), ("price_plus", "se_plus")):
        book = np.array([r["book"][est] for r in runs])
        ratio = np.mean([r["book"][se] for r in runs]) / book.std(ddof=1)
        x = np.array([r[est] for r in runs])
        rc = np.array([r[se] for r in runs]).mean(axis=0) / x.std(axis=0, ddof=1)
        print(f"{est}: book se / spread {ratio:.3f}, per option median {np.median(rc):.3f} [{rc.min():.3f}, {rc.max():.3f}]")
        assert 0.75 < ratio < 1.25, (est, ratio)
        assert 0.75 < np.median(rc) < 1.25, (est, np.median(rc))
        assert rc.min() > 0.55 and rc.max() < 1.6, (est, rc.min(), rc.max())


# ---------------------------------------------------------------- 8. split form
def test_split_form_and_reproducibility(engine, hw, curve):
    import torch
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    nq = 11 * (len(sw) + 1)
    full = torch.zeros(nq, dtype=torch.float64, device="cuda")
    a_part, b_part = torch.zeros_like(full), torch.zeros_like(full)
    a = 3 * 1024 + 17
    torch.cuda.synchronize()
    rng = hw.Rng(SEED + 5, N).seek(3)
    engine.swaptions_vega_moments(rng, sw, fl, P, f, full.data_ptr(), eps=EPS)
    assert rng.tell() == 3 + 900
    engine.swaptions_vega_moments(hw.Rng(SEED + 5, a).seek(3), sw, fl, P, f, a_part.data_ptr(), eps=EPS)
    engine.swaptions_vega_moments(hw.Rng(SEED + 5, N - a, first_path=a).seek(3), sw, fl, P, f, b_part.data_ptr(),
                                  eps=EPS)
    engine.synchronize()
    f_, s_ = full.cpu().numpy(), (a_part + b_part).cpu().numpy()
    assert np.allclose(f_, s_, rtol=2e-6, atol=0), np.abs(f_ / s_ - 1).max()
    fin = engine.swaptions_vega_finish(full.data_ptr(), N, sw, fl, P, eps=EPS)
    one_call = engine.swaptions_vega(hw.Rng(SEED + 5, N).seek(3), sw, fl, P, f, eps=EPS)
    same_result(fin, one_call)
    # the first 5 (n + 1) doubles are the swaptions_moments vector
    sm = torch.zeros(5 * (len(sw) + 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    engine.swaptions_moments(hw.Rng(SEED + 5, N).seek(3), sw, fl, P, f, sm.data_ptr())
    engine.synchronize()
    assert np.array_equal(sm.cpu().numpy(), f_[:5 * (len(sw) + 1)])
    again = engine.swaptions_vega(hw.Rng(SEED + 5, N).seek(3), sw, fl, P, f, eps=EPS)
    same_result(again, one_call)


# ---------------------------------------------------------------- 9. rejected arguments
def test_rejected_arguments(engine, hw, curve):
    P, f = curve["P"], curve["f"]
    sigma = float(engine.params.sigma)
    good = one(1.0, [(1.5, 0.02), (2.0, 1.02)], 1.0, 1.0)
    cases = [(name, book, EPS) for name, book in rejected_cases(engine, hw)]
    cases += [(f"eps {e}", good, e) for e in (0.0, -1e-3, np.nan, np.inf, -np.inf, sigma, 2 * sigma)]
    for name, (sw, fl), eps in cases:
        rng = hw.Rng(SEED, N).seek(7)
        before = engine.launch_count
        with pytest.raises(hw.HW1FError) as ei:
            engine.swaptions_vega(rng, sw, fl, P, f, eps=eps)
        assert ei.value.status == hw._ffi.ERR_INVALID, name
        assert len(str(ei.value).split(":", 1)[1].strip()) > 10, (name, str(ei.value))
        with pytest.raises(hw.HW1FError) as ei:
            engine.swaptions_vega_moments(rng, sw, fl, P, f, 0, eps=eps)
        assert ei.value.status == hw._ffi.ERR_INVALID, name
        assert engine.launch_count == before, name
        assert rng.tell() == 7, name
    with pytest.raises(hw.HW1FError) as ei:
        engine.cap_floor_vega(hw.Rng(SEED, N), caplets(hw, P, 10.0, n=3), P, f, kind="collar")
    assert ei.value.status == hw._ffi.ERR_INVALID


# ---------------------------------------------------------------- 10. edges
def test_never_paying_option(engine, hw, oracle, curve):
    P, f = curve["P"], curve["f"]
    sw, fl = merge(one(2.0, [(3.0, 0.03), (4.0, 1.03)], 0.01, 100.0, kind="payer"),
                   one(2.0, [(3.0, 0.03), (4.0, 1.03)], 5.0, 100.0, kind="receiver"),
                   one(6.0, [(7.0, 0.03), (8.0, 1.03)], 1.0, 100.0, kind="payer"))
    got = engine.swaptions_vega(hw.Rng(SEED + 3, N).seek(2), sw, fl, P, f, eps=EPS)
    for k in VEGA_KEYS:
        assert np.isfinite(got[k]).all(), k
        assert (np.asarray(got[k])[:2] == 0.0).all(), k
    assert all(np.isfinite(v).all() for v in got["book"].values())
    assert got["price_minus"][2] > 0 and got["vega"][2] > 0
    ref, aux = svo.vega_moments(oracle, SEED + 3, N, sw, fl, P, f, EPS, offset=2)
    check_vs_oracle(got, ref, aux, len(sw), what="never paying")


def test_exercise_at_first_and_last_step(engine, hw, oracle, curve):
    P, f = curve["P"], curve["f"]
    ns, Tf = engine.n_steps, float(engine.params.T_final)
    dt = Tf / ns
    sw, fl = merge(one(dt, [(0.5, 0.02), (1.0, 1.02)], 1.0, 10.0, kind="receiver", step=1),
                   one(Tf - dt, [(Tf, 1.0)], 0.9997, 10.0, kind="payer", step=ns))
    for off in (0, 1):
        rng = hw.Rng(SEED + 11, N).seek(off)
        got = engine.swaptions_vega(rng, sw, fl, P, f, eps=EPS)
        assert rng.tell() == off + ns
        ref, aux = svo.vega_moments(oracle, SEED + 11, N, sw, fl, P, f, EPS, offset=off)
        # one step from r0: test_gpu_swaption's allowance for 1-2 steps
        check_vs_oracle(got, ref, aux, len(sw), rel=2e-4, what=f"first and last step, offset {off}")


def test_smallest_model(engine, hw):
    from oracle_lib import Oracle
    over = dict(n_steps=2, n_mat=3, T_final=0.5)
    o = Oracle(**over)
    eng = engine_like(engine, hw, **over)
    try:
        n = 1 << 12
        c = eng.bond_curve(hw.Rng(31340, n))
        K = float(c["P"][2] / c["P"][1] * 1.0001 + 0.0001)
        sw, fl = merge(one(0.25, [(0.375, 0.0001), (0.5, 1.0)], K, 1.0, kind="payer"),
                       one(0.25, [(0.5, 1.0)], K, 1.0, kind="receiver"))
        for off in (0, 1):
            got = eng.swaptions_vega(hw.Rng(9, n).seek(off), sw, fl, c["P"], c["f"], eps=EPS)
            ref, aux = svo.vega_moments(o, 9, n, sw, fl, c["P"], c["f"], EPS, offset=off)
            check_vs_oracle(got, ref, aux, len(sw), rel=2e-4, what=f"2 x 3 model, offset {off}")
    finally:
        eng.close()


@pytest.mark.parametrize("n_steps", [1000, 8184])
def test_hundred_swaptions_2048_flows(engine, hw, n_steps):
    """HW1F_MAX_SWAPTIONS x HW1F_MAX_SWAPTION_FLOWS: decomposed mode must price it; reference order on 8184 steps
    stages three drift tables and may be refused, but only with HW1F_ERR_UNSUPPORTED before any launch"""
    from oracle_lib import Oracle
    over = dict(n_steps=n_steps, n_mat=n_steps // 8 + 1)
    o = Oracle(**over)
    eng = engine_like(engine, hw, **over)
    try:
        n, ns, Tf = 1 << 10, eng.n_steps, float(eng.params.T_final)
        c = eng.bond_curve(hw.Rng(31339, 1 << 12))
        sw, fl = hundred_on_longest(hw, c["P"], ns, Tf)
        rng = hw.Rng(8, n).seek(1)
        before = eng.launch_count
        try:
            got = eng.swaptions_vega(rng, sw, fl, c["P"], c["f"], eps=EPS)
        except hw.HW1FError as err:
            print(f"{n_steps} steps, {eng.mode}: refused: {err}")
            assert err.status == hw._ffi.ERR_UNSUPPORTED and "shared memory" in str(err)
            assert eng.mode == hw._ffi.MODE_REFERENCE_ORDER and n_steps == 8184
            assert rng.tell() == 1 and eng.launch_count == before
            return
        assert rng.tell() == 1 + int(sw["n_steps_exercise"][-1])
        ref, aux = svo.vega_moments(o, 8, n, sw, fl, c["P"], c["f"], EPS, offset=1)
        check_vs_oracle(got, ref, aux, len(sw), rel=5e-6, what=f"100 swaptions, 2048 flows, {n_steps} steps")
    finally:
        eng.close()


def test_new_entry_points_as_first_call_of_a_fresh_engine(engine, hw, curve):
    import torch
    P, f = curve["P"], curve["f"]
    sw, fl = mixed_book(hw, P)
    want = engine.swaptions_vega(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f, eps=EPS)
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        got = e.swaptions_vega(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f, eps=EPS)
    finally:
        e.close()
    same_result(got, want)
    mom = torch.zeros(11 * (len(sw) + 1), dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        e.swaptions_vega_moments(hw.Rng(SEED + 12, N + 5).seek(1), sw, fl, P, f, mom.data_ptr(), eps=EPS)
        e.synchronize()
        fin = e.swaptions_vega_finish(mom.data_ptr(), N + 5, sw, fl, P, eps=EPS)
    finally:
        e.close()
    same_result(fin, want)


def test_peer_mailbox_limit(engine, hw, curve):
    """with a (one-rank) communicator attached, 11 (n + 1) moments must fit the 512-double mailboxes: n <= 45"""
    import torch
    lib = hw._ffi.load()
    handle = (C.c_ubyte * 64)()
    h = C.c_void_p()
    e = hw.Engine(device=0)
    e.set_mode(engine.mode)
    try:
        if lib.hw1f_comm_create(e._h, 1, handle, C.byref(h)) != hw._ffi.OK:
            pytest.skip("no one-rank communicator on this machine")
        try:
            if lib.hw1f_comm_connect(h, 0, handle, None) != hw._ffi.OK or lib.hw1f_comm_attach(h, 1) != hw._ffi.OK:
                pytest.skip("a one-rank communicator cannot be attached here")
            P, f = curve["P"], curve["f"]
            sw, fl = hw.swaption_schedule(1.0 + 0.1 * np.arange(46), 2.0, 0.03, freq=2)     # expiries on the step grid
            mom = torch.zeros(11 * 47, dtype=torch.float64, device="cuda")
            torch.cuda.synchronize()
            rng = hw.Rng(SEED, N)
            before = e.launch_count
            with pytest.raises(hw.HW1FError) as ei:
                e.swaptions_vega_moments(rng, sw, fl, P, f, mom.data_ptr(), eps=EPS)
            assert ei.value.status == hw._ffi.ERR_INVALID and "45" in str(ei.value)
            assert rng.tell() == 0 and e.launch_count == before
            e.swaptions_vega_moments(rng, sw[:45], fl, P, f, mom.data_ptr(), eps=EPS)
            e.synchronize()
            assert rng.tell() > 0
            fin = e.swaptions_vega_finish(mom.data_ptr(), N, sw[:45], fl, P, eps=EPS)
            lib.hw1f_comm_attach(h, 0)
            want = e.swaptions_vega(hw.Rng(SEED, N), sw[:45], fl, P, f, eps=EPS)
            same_result(fin, want)
        finally:
            e.synchronize()
            lib.hw1f_comm_destroy(h)
    finally:
        e.close()


# ---------------------------------------------------------------- blocks that stride over several chunks
KCHUNK = 1024
MODEL = dict(n_steps=40, n_mat=11, T_final=0.4)   # dt 0.01
FIRST = 300
GS_SEED = 4247


def chunk_count(first, n):
    return (first + n - 1) // KCHUNK - first // KCHUNK + 1


def test_grid_stride_vs_oracle_and_shards(engine, hw):
    """(2 C + 37) * 1024 + 5 subsequences from path 300 (C = 32 x SM count, the grid cap): blocks run 2-3 chunks"""
    import torch
    from oracle_lib import Oracle
    grid = 32 * torch.cuda.get_device_properties(0).multi_processor_count
    n = (2 * grid + 37) * KCHUNK + 5
    assert 2 * grid < chunk_count(FIRST, n) < 3 * grid
    b1, b2 = (grid - 1) * KCHUNK, (2 * grid - 3) * KCHUNK + 517
    shards = [(FIRST, b1 - FIRST), (b1, b2 - b1), (b2, FIRST + n - b2)]
    assert all(chunk_count(f_, c) <= grid for f_, c in shards)
    o = Oracle(**MODEL)
    s, _ = o.bond_curve_sums(GS_SEED, 1 << 16)
    P, f = o.curve_finalize(s, 1 << 16)
    sw, fl = short_book(hw, P)
    e = engine_like(engine, hw, **MODEL)
    try:
        rng = hw.Rng(GS_SEED + 1, n, first_path=FIRST).seek(1)
        got = e.swaptions_vega(rng, sw, fl, P, f, eps=EPS)
        assert rng.tell() == 1 + 37
        ref, aux = svo.vega_moments(o, GS_SEED + 1, n, sw, fl, P, f, EPS, first_path=FIRST, offset=1)
        check_vs_oracle(got, ref, aux, len(sw), what="grid stride vs oracle")
        nq = 11 * (len(sw) + 1)
        full = torch.zeros(nq, dtype=torch.float64, device="cuda")
        acc, part = torch.zeros_like(full), torch.zeros_like(full)
        torch.cuda.synchronize()
        e.swaptions_vega_moments(hw.Rng(GS_SEED + 5, n, first_path=FIRST).seek(1), sw, fl, P, f, full.data_ptr(),
                                 eps=EPS)
        e.synchronize()
        for first, cnt in shards:
            e.swaptions_vega_moments(hw.Rng(GS_SEED + 5, cnt, first_path=first).seek(1), sw, fl, P, f, part.data_ptr(),
                                     eps=EPS)
            e.synchronize()
            acc += part
            torch.cuda.synchronize()          # the next launch overwrites `part`
    finally:
        e.close()
    a, b = full.cpu().numpy(), acc.cpu().numpy()
    assert np.isfinite(a).all()
    nz = a != 0
    rel = np.abs(a[nz] - b[nz]) / np.abs(a[nz])
    print(f"worst relative gap full vs shards {rel.max():.3g}")
    # float warp trees: a missing or doubled chunk moves a sum by ~1e-4 (test_gpu_grid_stride)
    assert (rel <= 1e-9).all() and (b[~nz] == 0).all(), rel.max()
