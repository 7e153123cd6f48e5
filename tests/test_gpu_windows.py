"""GPU: every solver entry on the window-edge fleets of tests/test_window_bands.py, bit for bit against the oracle.

Bit parity alone cannot see a wrong window bound: a solve that bails goes to the stored-vector fallback, which gives
the same bits, and a too-wide upper bound only changes which path computes them.  So the tests also check the path:
how many solves took the fallback (`wva_dbg_fallback_count`) and which grid rows shared their chain
(`wva_dbg_read_rows`), against what the band calculator predicts.

One bound is output-equivalent and no test here can tell it apart: pass 2's raised lower bound 2^(E(sum) - 960)
(`kHiPnSpan`).  It sends states with p / sum < 2^-960 to div.rn.f64 instead of the reciprocal division by the sum.
Below that ratio the reciprocal division can lose its low-word product to underflow, or return a subnormal quotient,
and be off by one unit in the last place.  That quotient is below 2^-960, yet it is only ever added to
`acc = sum(i p[i] / sum)`, at least 2^-24 (the normalised states sum to 1 over fewer than 2^23 states), and to `sumP`,
about 1, and rounded to float32 as p[K] / sum, which is 0 either way.  Every output bit is the same, and the bound
decides no bail, so the fallback count is the same too.  `tests/test_window_bands.py` still checks that the raised
band is reached (`n_raised`).
"""
import ctypes as C

import numpy as np
import pytest

from tests.bands import chain_bands, row_bands
from tests.test_window_bands import (NARROW_LAMBDA, RAISED_IDX, RAISED_N, RAISED_RATES, SHARP_IDX, SHARP_N,
                                     SHARP_RATES, WIDE_N, _analyzer, f32, grid_lambda, narrow_fleet, narrow_grid,
                                     overflow_fleet, raised_fleet, rate_edge_fleet, sharp_peak_fleet, sweep_lambdas,
                                     wide_fleet)
from tests.util import assert_allocs_equal, assert_f32_bits_equal

pytestmark = pytest.mark.gpu


def _fallbacks(engine):
    L = engine._L
    L.wva_dbg_fallback_count.restype = C.c_int
    L.wva_dbg_fallback_count.argtypes = [C.c_void_p]
    return int(L.wva_dbg_fallback_count(engine._h))


def _rows(engine):
    L = engine._L
    L.wva_dbg_read_rows.restype = C.c_longlong
    L.wva_dbg_read_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
    cap = 1 << 16
    row_j = np.zeros(cap, np.int32)
    res = np.zeros(cap, np.uint8)
    n = L.wva_dbg_read_rows(engine._h, row_j.ctypes.data, res.ctypes.data, cap)
    return row_j[:n], res[:n]


# ---- grid_solve / grid_rows / solve_row -------------------------------------------------------------------------
@pytest.mark.parametrize("rowres", [0, 1])
@pytest.mark.parametrize("want_cells", [False, True])
def test_grid_narrow_edges(engine, oracle_mod, monkeypatch, rowres, want_cells):
    fleet, grid = narrow_fleet(), narrow_grid()
    monkeypatch.setenv("WVA_GRID_ROWRES", str(rowres))
    cells_o, win_o = oracle_mod.grid_solve(fleet, grid, want_cells=True)
    cells_g, win_g = engine.grid_solve(fleet, grid, want_cells=want_cells)
    n_fb = _fallbacks(engine)
    row_j, _ = _rows(engine)
    assert_allocs_equal(win_g, win_o, "grid winners")
    if want_cells:
        assert np.array_equal(cells_g["flags"], cells_o["flags"]), "cell flags"
        for k in ("ttft", "itl", "rho", "throughput"):
            assert_f32_bits_equal(cells_g[k], cells_o[k], f"cells.{k}")
    # the rows: shared exactly where the calculator says (a sum of 2^620 or more is never shared)
    bmax = int(max(grid.batch))
    R = grid.replicas.size
    n_above = 0
    for s in range(fleet.n_servers):
        sr = _analyzer(fleet, s, bmax).serv_rate()
        for ri, r in enumerate(grid.replicas):
            b = row_bands(sr, bmax, grid_lambda(fleet, s, int(r)))
            shared = row_j[s * R + ri] != np.iinfo(np.int32).max
            assert shared == b["shared"], f"row lambda {NARROW_LAMBDA[s]}/{r}: shared {shared}, sum 2^{b['e_sum']}"
            n_above += b.get("sum_ok") is False
    assert n_above >= 2
    # every analysable cell whose chain leaves the narrow windows (peak 2^600, sum 2^620) and does not share its row's
    # chain takes the fallback (row resolution only skips cells that share the chain)
    want = 0
    for s in range(fleet.n_servers):
        sr = _analyzer(fleet, s, bmax).serv_rate()
        for ri, r in enumerate(grid.replicas):
            lam = grid_lambda(fleet, s, int(r))
            row_shared = row_j[s * R + ri] != np.iinfo(np.int32).max
            for b in grid.batch:
                b = int(b)
                rmax = f32(f32(f32(sr[b - 1]) * f32(1 - f32(0.001))) * f32(1000))
                if not f32(lam * f32(1000)) <= rmax:
                    continue
                if row_shared and b >= row_j[s * R + ri] + 2:
                    continue
                c = chain_bands(sr, b, 11 * b, lam)
                want += c["e_peak"] >= 600 or c["e_sum"] >= 620
    assert n_fb == want > 0, f"fallback cells {n_fb}, predicted {want}"


# ---- analyze / solve: size_warp_kernel and the rounds path ---------------------------------------------------
def _size_expect(fleet):
    """Candidates whose Size evaluations include one outside the wide windows: with the linear fleets, the largest
    lambda is RateRange.Max/1000, so a candidate bails exactly when that chain does."""
    n = 0
    for s in range(fleet.n_servers):
        N = int(fleet.srv_max_batch[s])
        qa = _analyzer(fleet, s, N)
        lmax = f32(f32(qa.rate_range()[1]) / f32(1000))
        b = chain_bands(qa.serv_rate(), N, qa.K, lmax)
        n += (not b["rates_ok"]) or b["e_peak"] >= 880 or b["e_sum"] >= 900
    return n


@pytest.mark.parametrize("path", ["warp", "rounds-d1", "rounds-d5"])
def test_size_wide_edges(engine, oracle_mod, monkeypatch, path):
    monkeypatch.setenv("WVA_SIZE_SMALL_MAX", "100000" if path == "warp" else "0")
    if path != "warp":
        monkeypatch.setenv("WVA_SIZE_DEPTH", path[-1])
    for name, fleet in (("wide", wide_fleet()), ("raised", raised_fleet()), ("rate_edge", rate_edge_fleet()),
                        ("overflow", overflow_fleet())):
        cand_o, win_o = oracle_mod.solve(fleet)
        cand_g, win_g = engine.solve(fleet)
        assert_allocs_equal(cand_g, cand_o, f"{name}: size candidates ({path})")
        assert_allocs_equal(win_g, win_o, f"{name}: winners ({path})")
        if name != "overflow":
            assert _fallbacks(engine) == _size_expect(fleet), f"{name}: fallback candidates ({path})"
        assert_allocs_equal(engine.analyze(fleet), oracle_mod.calculate(fleet), f"{name}: analyze ({path})")
    # the wide fleet bails from N = 615 on (peak 2^880) and not below it (N = 614: peak 2^878, sum 2^888)
    assert _size_expect(wide_fleet()) == sum(N >= 615 for N in WIDE_N)
    assert _size_expect(rate_edge_fleet()) == 4   # servRate 2^60, lambda 0.999 * 2^-60 twice, lambda below 2^-60


# ---- upload + update_load + resolve ---------------------------------------------------------------------------
def test_resolve_ticks_across_the_edge(engine, oracle_mod):
    """N = 640 at one replica: ticks move CreateAllocation's final lambda (total rate / replicas) across the lambda
    where the peak reaches 2^880 and back."""
    fleet = wide_fleet().take_servers(np.array([WIDE_N.index(640)]))
    fleet.srv_slo_ttft[:] = 1e6
    qa = _analyzer(fleet, 0, 640)
    sr = qa.serv_rate()
    lo, hi = 560.0, 639.0
    for _ in range(30):   # the lambda where the peak first reaches 2^880
        mid = (lo + hi) / 2
        if chain_bands(sr, 640, qa.K, f32(mid))["e_peak"] >= 880:
            hi = mid
        else:
            lo = mid
    edge = hi
    ticks = [edge * 0.999, edge * 1.001, edge * 0.998, edge * 1.01]
    engine.upload(fleet)
    seen = set()
    for lam in ticks:
        fleet.srv_arrival_rpm[:] = np.float32(lam * 60000.0)
        engine.update_load(arrival_rpm=fleet.srv_arrival_rpm)
        _, win_g = engine.resolve()
        _, win_o = oracle_mod.solve(fleet)
        assert_allocs_equal(win_g, win_o, f"resolve at lambda {lam}")
        rec = oracle_mod.create_allocation(fleet, 0, 0)
        seen.add(chain_bands(sr, 640, qa.K, grid_lambda(fleet, 0, rec["replicas"]))["e_peak"] >= 880)
    assert seen == {False, True}, "the ticks must put the final Analyze on both sides of the edge"


# ---- sweep ---------------------------------------------------------------------------------------------------
def _sweep_check(engine, oracle_mod, fleet, n_rates, what):
    o = oracle_mod.sweep(fleet, n_rates)
    g = engine.sweep(fleet, n_rates)
    assert np.array_equal(g["valid"], o["valid"]), f"{what}: valid"
    for k in ("rate", "ttft", "itl", "throughput", "rho"):
        assert_f32_bits_equal(g[k], o[k], f"{what}: sweep.{k}")
    return o


def _sweep_expect(fleet, n_rates):
    n = 0
    for s in range(fleet.n_servers):
        N = int(fleet.srv_max_batch[s])
        qa = _analyzer(fleet, s, N)
        for lam in sweep_lambdas(*qa.rate_range(), n_rates):
            b = chain_bands(qa.serv_rate(), N, qa.K, lam)
            n += (not b["rates_ok"]) or b["e_peak"] >= 880 or b["e_sum"] >= 900
    return n


def test_sweep_wide_edges(engine, oracle_mod):
    fleet = wide_fleet()
    o = _sweep_check(engine, oracle_mod, fleet, 64, "wide")
    assert o["valid"].all()
    assert _fallbacks(engine) == _sweep_expect(fleet, 64) > 0
    fleet = rate_edge_fleet()
    _sweep_check(engine, oracle_mod, fleet, 8, "rate edge")
    assert _fallbacks(engine) == _sweep_expect(fleet, 8) > 0


def test_sweep_block_straddles_sharp_peak(engine, oracle_mod):
    """The narrow peak of sharp_peak_fleet: the solver must bail on every sweep index of SHARP_IDX although a 4-step
    block without the 3 e_hi margin would step over the peak and stream to the same bits."""
    fleet = sharp_peak_fleet()
    _sweep_check(engine, oracle_mod, fleet, SHARP_RATES, "sharp peak")
    qa = _analyzer(fleet, 0, SHARP_N)
    lams = sweep_lambdas(*qa.rate_range(), SHARP_RATES)
    for i in SHARP_IDX:
        b = chain_bands(qa.serv_rate(), SHARP_N, qa.K, lams[i])
        assert b["block_straddle"] and b["e_hi"] > 0 and b["e_sum"] < 900, i
    assert _fallbacks(engine) == _sweep_expect(fleet, SHARP_RATES)


def test_sweep_raised_band(engine, oracle_mod):
    fleet = raised_fleet()
    _sweep_check(engine, oracle_mod, fleet, RAISED_RATES, "raised")
    qa = _analyzer(fleet, 0, RAISED_N)
    lams = sweep_lambdas(*qa.rate_range(), RAISED_RATES)
    for i in RAISED_IDX:   # these stream (no bail) through the raised pass-2 band
        b = chain_bands(qa.serv_rate(), RAISED_N, qa.K, lams[i])
        assert b["n_raised"] > 0 and b["e_peak"] < 880, i
    assert _fallbacks(engine) == _sweep_expect(fleet, RAISED_RATES)


@pytest.mark.parametrize("case", ["n640", "overflow_n1024"])
def test_sweep_falls_back_to_stored_vector(engine, oracle_mod, case):
    """Sweep points whose chain leaves the streaming windows (N = 640 near RateRange.Max: sum above 2^900; N = 1024:
    overflow, the reference rescales) are re-run on the stored-vector fallback instead of failing the call."""
    fleet = (wide_fleet().take_servers(np.array([WIDE_N.index(640)])) if case == "n640" else overflow_fleet())
    o = _sweep_check(engine, oracle_mod, fleet, 32, case)
    assert o["valid"].all()
    assert _fallbacks(engine) > 0
