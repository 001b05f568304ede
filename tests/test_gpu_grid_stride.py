"""Runs in which every simulation block strides over two or three chunks.

Every simulation kernel loops `for (chunk = blockIdx.x; chunk < n_chunks; chunk += gridDim.x)` over chunks of kChunk =
1024 subsequences, on a grid capped at 32 blocks per SM.  The large production runs (2^27 subsequences per GPU) give
each block ~28 chunks, so the block accumulators, the per-chunk state that must be reset, the stream derivation of the
second and later chunks, the parked noise state of the recalibrated FD pass and the per-block path counts of the batch
means all matter there.  These tests size the run from the device so that the chunk count exceeds twice the grid, and
check it against the CPU oracle, against the sum of shards that each fit in one grid pass, across entry points, and
through the batch-means standard errors."""
import numpy as np
import pytest

import cap_oracle
from cap_closed_form import atm_rate

pytestmark = pytest.mark.gpu

KCHUNK = 1024                                # kChunk = 2 * kThreads subsequences per block pass
MODEL = dict(n_steps=40, n_mat=11, T_final=0.4)   # dt 0.01, save stride 4: S1 = 0.2 is maturity 5 (the fused pass needs that)
S1, S2, NS1 = 0.2, 0.4, 20
FIRST = 300                                  # unaligned: the first chunk of every run is ragged
SEED = 4242
# reset steps of the strip: gaps 1, 3, 4, 0 (two caplets on one step), 9, 2, 5, 7, 6
CAP_STEPS = np.array([1, 4, 8, 8, 17, 19, 24, 31, 37])
CAP_TAU = np.array([0.02, 0.03, 0.02, 0.04, 0.02, 0.03, 0.02, 0.05, 0.02])


def chunk_count(first, n):
    return (first + n - 1) // KCHUNK - first // KCHUNK + 1


@pytest.fixture(scope="module")
def geom():
    import torch
    grid = 32 * torch.cuda.get_device_properties(0).multi_processor_count      # prepare_launch's grid cap
    n = (2 * grid + 37) * KCHUNK + 5
    n_chunks = chunk_count(FIRST, n)
    # every block runs 2 or 3 chunks; if the grid or the chunk size changes, this fails instead of going stale
    assert 2 * grid < n_chunks < 3 * grid, (grid, n_chunks)
    assert FIRST % KCHUNK and (FIRST + n) % KCHUNK          # both edge chunks ragged
    # shards of at most `grid` chunks each (one grid pass): one boundary chunk-aligned, one inside a chunk
    b1 = (grid - 1) * KCHUNK
    b2 = (2 * grid - 3) * KCHUNK + 517
    shards = [(FIRST, b1 - FIRST), (b1, b2 - b1), (b2, FIRST + n - b2)]
    assert all(chunk_count(f, c) <= grid for f, c in shards)
    print(f"grid {grid} blocks, {n} subsequences from {FIRST}: {n_chunks} chunks, "
          f"{n_chunks - 2 * grid} blocks of 3 chunks / {3 * grid - n_chunks} of 2")
    return dict(grid=grid, n=n, n_chunks=n_chunks, shards=shards)


def strip(hw, P):
    resets = CAP_STEPS * 0.01
    pays = resets + CAP_TAU
    caps = hw.caplet_schedule(resets, pays, atm_rate(P, resets, pays, MODEL["T_final"]))
    caps["n_steps_reset"] = CAP_STEPS
    return caps


@pytest.fixture(scope="module")
def ref(geom, hw):
    """oracle results at the full size, shared by both modes (the per-path jump-ahead dominates: ~15 s per call)"""
    from oracle_lib import Oracle
    o = Oracle(**MODEL)
    n = geom["n"]
    s, _ = o.bond_curve_sums(SEED, n, first_path=FIRST)
    P, f = o.curve_finalize(s, n)
    K = float(np.float32(0.9) * P[10] / P[5])      # test_other_model_parameters' strike: almost every path pays
    caps = strip(hw, P)
    return dict(
        P=P, f=f, K=K, caps=caps,
        zbc=o.zbc_moments(SEED + 1, n, P, f, S1=S1, S2=S2, K=K, n_steps_S1=NS1, first_path=FIRST),
        vega=o.vega_pathwise_sums(SEED + 2, n, P, f, S1=S1, S2=S2, K=K, n_steps_S1=NS1, first_path=FIRST),
        cap=cap_oracle.cap_moments(o, SEED + 3, n, caps, P, f, kind="cap", first_path=FIRST, offset=1))


@pytest.fixture(scope="module")
def short(engine, hw):
    e = hw.Engine(device=0, params=hw.default_params(**MODEL))
    e.set_mode(engine.mode)
    yield e
    e.close()


def rng(hw, seed, first, n, offset=0):
    return hw.Rng(seed, n, first_path=first).seek(offset)


# ---------------------------------------------------------------- 1. against the oracle
def test_full_size_vs_oracle(short, hw, geom, ref):
    n = geom["n"]
    P, f, K = ref["P"], ref["f"], ref["K"]
    # a dropped or doubled chunk moves every sum by ~1 / n_chunks = 1e-4 relative: far outside each bound below
    c = short.bond_curve(rng(hw, SEED, FIRST, n))
    assert np.abs(c["P"] / P - 1).max() < 1e-6 and np.abs(c["f"] - f).max() < 5e-6      # test_tiny_and_ragged_path_counts
    z = short.zbc_cv(rng(hw, SEED + 1, FIRST, n), P, f, S1=S1, S2=S2, K=K, n_steps_S1=NS1)
    assert np.allclose(z["mom"], ref["zbc"], rtol=5e-6), (z["mom"], ref["zbc"])            # test_other_model_parameters
    v = short.vega_pathwise(rng(hw, SEED + 2, FIRST, n), P, f, S1=S1, S2=S2, K=K, n_steps_S1=NS1)
    assert v["vega_pathwise_f64"] == pytest.approx(ref["vega"][0] / n, rel=2e-5, abs=1e-7)
    r = rng(hw, SEED + 3, FIRST, n, offset=1)          # odd offset: every chunk starts on a cached cos half
    cp = short.cap_floor(r, ref["caps"], P, f, kind="cap")
    assert r.tell() == 1 + CAP_STEPS[-1]
    mom = np.vstack([cp["mom"], np.asarray(cp["strip"]["mom"])[None, :]])
    gap, bound = np.abs(mom - ref["cap"]), cap_oracle.moment_bound(ref["cap"])      # test_cap_moments_vs_oracle
    print(f"strip: worst moment gap / bound {(gap / bound).max():.3g}")
    assert (gap <= bound).all(), np.unravel_index((gap / bound).argmax(), gap.shape)


# ---------------------------------------------------------------- 2. full run == sum of one-pass shards
# What the bounds must separate: one missing or duplicated chunk out of ~9500 moves a sum by ~1e-4 relative.  What
# they must allow: the order of the double accumulation (block accumulators, tail) moves it by ~1e-14, and where a
# kernel sums through float warp trees, the one chunk a ragged shard boundary straddles is grouped differently: a
# float rounding of ~1e-7 of one chunk's (centred, for the curve and the caplet controls) contribution, < 1e-10 of the
# total.  So 1e-12 where the partials are double from the per-path values on, 1e-9 where they pass float warp trees.
TIGHT, FLOAT_TREES = 1e-12, 1e-9


def _entry(short, ref, which, nm, n_caps):
    P, f, K = ref["P"], ref["f"], ref["K"]
    kw = dict(S1=S1, S2=S2, K=K, n_steps_S1=NS1)
    curve = [(slice(1, nm), FLOAT_TREES), (slice(nm + 1, 2 * nm), FLOAT_TREES)]   # P(0) = 1 is not simulated
    if which == "bond_curve":
        return 2 * nm, lambda r, p: short.bond_curve_moments(r, p), curve
    if which == "zbc_cv":
        return 5, lambda r, p: short.zbc_cv_moments(r, P, f, p, **kw), [(slice(0, 5), TIGHT)]
    if which == "vega_pathwise":
        return 2, lambda r, p: short.vega_pathwise_moments(r, P, f, p, **kw), [(slice(0, 2), TIGHT)]
    if which == "fused":
        return 2 * nm + 8, lambda r, p: short.fused_moments(r, P, f, p, **kw), curve + [(slice(2 * nm, None), TIGHT)]
    if which == "fused_fd":
        return (2 * nm + 18, lambda r, p: short.fused_moments(r, P, f, p, eps=0.001, **kw),
                curve + [(slice(2 * nm, None), TIGHT)])
    nq = 5 * (n_caps + 1)
    return nq, lambda r, p: short.cap_floor_moments(r, ref["caps"], P, f, p, kind="floor"), [(slice(0, nq), FLOAT_TREES)]


@pytest.mark.parametrize("which", ["bond_curve", "zbc_cv", "vega_pathwise", "fused", "fused_fd", "cap_floor"])
def test_full_run_equals_sum_of_shards(short, hw, geom, ref, which):
    import torch
    nq, call, checks = _entry(short, ref, which, short.n_mat, len(ref["caps"]))
    offset = 1 if which == "cap_floor" else 0
    full = torch.zeros(nq, dtype=torch.float64, device="cuda")
    acc, part = torch.zeros_like(full), torch.zeros_like(full)
    torch.cuda.synchronize()
    call(rng(hw, SEED + 5, FIRST, geom["n"], offset), full.data_ptr())
    short.synchronize()
    for first, cnt in geom["shards"]:
        call(rng(hw, SEED + 5, first, cnt, offset), part.data_ptr())
        short.synchronize()
        acc += part
        torch.cuda.synchronize()          # the next launch overwrites `part`
    a, b = full.cpu().numpy(), acc.cpu().numpy()
    assert np.isfinite(a).all()
    for sl, rtol in checks:
        rel = np.abs(a[sl] - b[sl]) / np.abs(a[sl])
        print(f"{which} {sl}: worst relative gap full vs shards {rel.max():.3g} (bound {rtol:g})")
        assert (rel <= rtol).all(), (which, sl, rel.max())


# ---------------------------------------------------------------- 3. identities across entry points
def test_fused_equals_separate_calls(short, hw, geom, ref):
    n, P, f, K = geom["n"], ref["P"], ref["f"], ref["K"]
    kw = dict(S1=S1, S2=S2, K=K, n_steps_S1=NS1)
    fu = short.fused(rng(hw, SEED + 6, FIRST, n), P, f, eps=0.001, **kw)
    c = short.bond_curve(rng(hw, SEED + 6, FIRST, n))
    assert (fu["P"] == c["P"]).all() and (fu["f"] == c["f"]).all()
    z = short.zbc_cv(rng(hw, SEED + 6, FIRST, n), P, f, **kw)
    assert fu["zbc"]["mom"] == z["mom"]
    fd = short.vega_fd(rng(hw, SEED + 6, FIRST, n), P, f, eps=0.001, **kw)
    assert fu["vega"]["price_minus"] == fd["price_minus"] and fu["vega"]["price_plus"] == fd["price_plus"]


def test_vega_fd_recalibrated_equals_bumped_engines(short, hw, geom, ref):
    """on the maturity grid the decomposed mode prices from the noise state the curve pass parked per chunk"""
    n, K, eps = geom["n"], ref["K"], 0.001
    kw = dict(S1=S1, S2=S2, K=K, n_steps_S1=NS1)
    got = short.vega_fd_recalibrated(rng(hw, SEED + 7, FIRST, n), eps=eps, **kw)
    prices = []
    for sgn in (-1.0, 1.0):
        e2 = hw.Engine(device=0, params=hw.default_params(sigma=float(np.float32(0.1) + np.float32(sgn * eps)), **MODEL))
        e2.set_mode(short.mode)
        try:
            c = e2.bond_curve(rng(hw, SEED + 7, FIRST, n))
            prices.append(e2.zbc_cv(rng(hw, SEED + 7, FIRST, n), c["P"], c["f"], **kw)["price_cv"])
        finally:
            e2.close()
    # the bound of test_vega_fd_recalibrated_equals_bumped_engines; one chunk on the wrong noise state moves a price
    # by its Monte Carlo noise, ~1e-4 relative at this strike
    assert got["price_minus_recal"] == pytest.approx(prices[0], rel=2e-6)
    assert got["price_plus_recal"] == pytest.approx(prices[1], rel=2e-6)


def test_batch_equals_single_runs(short, hw, geom, ref):
    n, P, f = geom["n"], ref["P"], ref["f"]
    assert chunk_count(0, n) > 2 * geom["grid"]
    kw = dict(S1=S1, S2=S2, K=ref["K"], n_steps_S1=NS1)
    res, _ = short.zbc_cv_batch([SEED + 8, SEED + 9], n, P, f, **kw)
    for s, r in zip([SEED + 8, SEED + 9], res):
        assert r["mom"] == short.zbc_cv(hw.Rng(s, n), P, f, **kw)["mom"], s


# ---------------------------------------------------------------- 4. batch means with unequal blocks
def test_batch_means_se_with_unequal_blocks(short, hw, geom):
    """bond_curve_ci weights each block's batch by the subsequences it simulated (block_subsequences): here 3 chunks
    for some blocks, 2 for the others, ragged at both ends.  A wrong count offsets a block's sum by ~1000 mean
    values and inflates P_se_batch by orders of magnitude."""
    c = short.bond_curve(rng(hw, SEED + 10, FIRST, geom["n"]))
    ci = short.bond_curve_ci()
    # test_gpu_ci._first_maturity: below T = 0.1 (decomposed) / 0.3 (reference order) the spread is float quantisation
    m0 = 3 if short.mode == hw._ffi.MODE_DECOMPOSED else 8
    exact, batch = c["P_se"][m0:].astype(np.float64), ci["P_se_batch"][m0:].astype(np.float64)
    assert (exact > 0).all()
    # the bound of test_P_se_exact_and_batch_means; with one batch per block (32 per SM) the estimate itself is good to ~1 %
    assert np.abs(batch / exact - 1).max() < 0.15, batch / exact
