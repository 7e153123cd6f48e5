"""GPU: wva_resolve_scenarios, block by block, against the oracle and against update_load + resolve on the device."""
import ctypes as C

import numpy as np
import pytest

from tests.scenarios import scenario_fleets, scenario_rows, with_arrival
from tests.test_window_bands import (WIDE_N, _analyzer, grid_lambda, overflow_fleet, raised_fleet, rate_edge_fleet,
                                     sharp_peak_fleet, wide_fleet)
from tests.bands import chain_bands
from tests.util import ALLOC_FIELDS, assert_allocs_equal, bits
from workload_variant_autoscaler_b200 import Engine, WvaError, _abi, synth_fleet

pytestmark = pytest.mark.gpu


class _Block:
    """Records lo .. hi - 1 of an Allocs, shaped like one (for tests.util.assert_allocs_equal)."""

    def __init__(self, allocs, lo, hi):
        self.n = hi - lo
        for f in ALLOC_FIELDS:
            setattr(self, f, getattr(allocs, f)[lo:hi])

    def record(self, i):
        return {f: getattr(self, f)[i].item() for f in ALLOC_FIELDS}


def _same(got, want, what):
    """Device records against device records, bit for bit."""
    assert got.n == want.n, what
    for f in ALLOC_FIELDS:
        g, w = getattr(got, f), getattr(want, f)
        bad = np.nonzero(bits(g) != bits(w))[0] if g.dtype == np.float32 else np.nonzero(g != w)[0]
        if bad.size:
            i = int(bad[0])
            raise AssertionError(f"{what}: {f}: {bad.size} of {got.n} differ; first at {i}\n got  {got.record(i)}\n"
                                 f" want {want.record(i)}")


def _fallbacks(engine):
    L = engine._L
    L.wva_dbg_fallback_count.restype = C.c_int
    L.wva_dbg_fallback_count.argtypes = [C.c_void_p]
    return int(L.wva_dbg_fallback_count(engine._h))


def _blocks(fleet, cand, win, l):
    SA, S = fleet.n_servers * fleet.n_acc, fleet.n_servers
    return _Block(cand, l * SA, (l + 1) * SA), _Block(win, l * S, (l + 1) * S)


def _plain(engine, row):
    engine.update_load(arrival_rpm=row)
    return engine.resolve(want_candidates=True)


def _check(engine, oracle_mod, fleet, rows, what, *, oracle=True):
    """One scenario call; every block against update_load + resolve and (optionally) the oracle.  Returns the rows
    where the plain device path itself differs from the oracle (those are compared device against device only)."""
    engine.upload(fleet)
    cand, win = engine.resolve_scenarios(rows, want_candidates=True)
    n_fb = _fallbacks(engine)
    plain_differs, plain_fb = [], 0
    for l, row in enumerate(rows):
        c, w = _blocks(fleet, cand, win, l)
        pc, pw = _plain(engine, row)
        plain_fb += _fallbacks(engine)
        _same(c, pc, f"{what} row {l}: candidates vs update_load + resolve")
        _same(w, pw, f"{what} row {l}: winners vs update_load + resolve")
        if not oracle:
            continue
        co, wo = oracle_mod.solve(with_arrival(fleet, row))
        try:
            assert_allocs_equal(pc, co, "plain")
            assert_allocs_equal(pw, wo, "plain")
        except AssertionError:
            plain_differs.append(l)
            continue
        assert_allocs_equal(c, co, f"{what} row {l}: candidates vs oracle")
        assert_allocs_equal(w, wo, f"{what} row {l}: winners vs oracle")
    return plain_differs, (n_fb, plain_fb)


@pytest.mark.parametrize("L", [1, 3, 17])
@pytest.mark.parametrize("name", ["plain", "keep", "gaps"])
def test_blocks_match_oracle_and_resolve(engine, oracle_mod, name, L):
    fleet = scenario_fleets()[name]
    rows = scenario_rows(fleet.srv_arrival_rpm, L, seed=L)
    differs, _ = _check(engine, oracle_mod, fleet, rows, f"{name} L={L}")
    # only rows with rates of 1e15 and above may push numReplicas past the int32 records on the plain path
    assert all((rows[l] >= 1e15).any() for l in differs), f"plain path differs from the oracle on rows {differs}"


def test_single_base_row_is_resolve(engine):
    fleet = scenario_fleets()["keep"]
    engine.upload(fleet)
    pc, pw = engine.resolve(want_candidates=True)
    cand, win = engine.resolve_scenarios(fleet.srv_arrival_rpm[None, :], want_candidates=True)
    _same(cand, pc, "L=1 candidates")
    _same(win, pw, "L=1 winners")


@pytest.mark.parametrize("small_max", ["0", None])
def test_both_size_paths(engine, oracle_mod, monkeypatch, small_max):
    """More than 1024 candidates: the plain resolve runs the warp kernel (default) or the rounds (0)."""
    if small_max is not None:
        monkeypatch.setenv("WVA_SIZE_SMALL_MAX", small_max)
    fleet = synth_fleet(300, 4, seed=9, max_batch_choices=(4, 8, 16, 32))
    rows = scenario_rows(fleet.srv_arrival_rpm, 4, seed=2)
    engine.upload(fleet)
    cand, win = engine.resolve_scenarios(rows, want_candidates=True)
    for l, row in enumerate(rows):
        c, w = _blocks(fleet, cand, win, l)
        pc, pw = _plain(engine, row)
        _same(c, pc, f"row {l} candidates")
        _same(w, pw, f"row {l} winners")
    co, wo = oracle_mod.solve(with_arrival(fleet, rows[1]))
    assert_allocs_equal(_blocks(fleet, cand, win, 1)[0], co, "row 1 candidates vs oracle")
    assert_allocs_equal(_blocks(fleet, cand, win, 1)[1], wo, "row 1 winners vs oracle")


@pytest.mark.parametrize("depth", ["1", "5"])
def test_depths(engine, oracle_mod, monkeypatch, depth):
    monkeypatch.setenv("WVA_SIZE_DEPTH", depth)
    fleet = scenario_fleets()["gaps"]
    rows = scenario_rows(fleet.srv_arrival_rpm, 9, seed=5)
    differs, _ = _check(engine, oracle_mod, fleet, rows, f"depth {depth}")
    assert all((rows[l] >= 1e15).any() for l in differs)


@pytest.mark.parametrize("policy", [0, 1, 2, 3])
def test_limited_mode(engine, oracle_mod, policy):
    fleet = synth_fleet(24, 4, seed=13, max_batch_choices=(4, 8, 16, 32), tps_frac=0.2)
    fleet.unlimited = False
    fleet.saturation_policy = policy
    fleet.delayed_best_effort = policy == 2
    fleet.type_capacity[:] = 24
    rows = scenario_rows(fleet.srv_arrival_rpm, seed=policy)[[0, 1, 2, 3, 4, 6, 13, 14, 16]]
    differs, _ = _check(engine, oracle_mod, fleet, rows, f"limited policy {policy}")
    assert differs == []


# ---- window-edge fleets -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["wide", "raised", "rate_edge", "overflow", "sharp_peak"])
def test_window_edge_fleets(engine, oracle_mod, name):
    fleet = {"wide": wide_fleet, "raised": raised_fleet, "rate_edge": rate_edge_fleet, "overflow": overflow_fleet,
             "sharp_peak": sharp_peak_fleet}[name]()
    base = fleet.srv_arrival_rpm
    rows = np.stack([base, base * np.float32(0.5), base * np.float32(0.999), base * np.float32(2)])
    engine.solve(fleet, want_candidates=False)
    base_fb = _fallbacks(engine)
    differs, (n_fb, plain_fb) = _check(engine, oracle_mod, fleet, rows, name)
    assert differs == []
    # a (candidate, scenario) takes the fallback exactly where that scenario's resolve does
    assert n_fb == plain_fb, f"{name}: {n_fb} fallback solves, {plain_fb} over the scenarios' resolves"
    if base_fb > 0:
        assert n_fb > 0, f"{name}: the base solve takes the fallback {base_fb} times, the scenarios never"


def test_final_analyze_across_the_edge(engine, oracle_mod):
    """N = 640 at one replica: the scenario rows put CreateAllocation's final lambda on both sides of the lambda where
    the chain's peak reaches 2^880 (bail to the stored-vector fallback above it)."""
    fleet = wide_fleet().take_servers(np.array([WIDE_N.index(640)]))
    fleet.srv_slo_ttft[:] = 1e6
    qa = _analyzer(fleet, 0, 640)
    sr = qa.serv_rate()
    lo, hi = 560.0, 639.0
    for _ in range(30):
        mid = (lo + hi) / 2
        if chain_bands(sr, 640, qa.K, np.float32(mid))["e_peak"] >= 880:
            hi = mid
        else:
            lo = mid
    rows = np.array([[hi * f * 60000.0] for f in (0.999, 1.001, 0.998, 1.01)], np.float32)
    above = 0
    for row in rows:
        f = with_arrival(fleet, row)
        rec = oracle_mod.create_allocation(f, 0, 0)
        above += chain_bands(sr, 640, qa.K, grid_lambda(f, 0, rec["replicas"]))["e_peak"] >= 880
    assert 0 < above < len(rows), "the rows must put the final Analyze on both sides of the edge"
    differs, (n_fb, plain_fb) = _check(engine, oracle_mod, fleet, rows, "edge")
    assert differs == []
    assert n_fb == plain_fb >= above, f"{n_fb} fallback solves, {plain_fb} over the resolves, {above} rows above"


# ---- state and errors --------------------------------------------------------------------------------------------
def test_nan_row_fails_like_solve(engine, oracle_mod):
    fleet = scenario_fleets()["plain"]
    rows = scenario_rows(fleet.srv_arrival_rpm, 3)
    bad = rows.copy()
    bad[1, ::2] = np.nan
    try:
        _, want = engine.solve(with_arrival(fleet, bad[1]), want_candidates=False)
        code = 0
    except WvaError as exc:
        code = exc.code
    engine.upload(fleet)
    if code:
        with pytest.raises(WvaError) as ei:
            engine.resolve_scenarios(bad)
        assert ei.value.code == code
    else:
        _, win = engine.resolve_scenarios(bad)
        _same(_Block(win, fleet.n_servers, 2 * fleet.n_servers), want, "NaN row winners")
    # the handle keeps working
    differs, _ = _check(engine, oracle_mod, fleet, rows, "after NaN")
    assert differs == []


def test_resident_fleet_unchanged(engine):
    fleet = scenario_fleets()["gaps"]
    engine.upload(fleet)
    pc, pw = engine.resolve(want_candidates=True)
    engine.summarize(fleet.n_types)
    engine.resolve_scenarios(scenario_rows(fleet.srv_arrival_rpm, 5) * np.float32(3))
    with pytest.raises(WvaError) as ei:
        engine.summarize(fleet.n_types)
    assert ei.value.code == _abi.WVA_ERR_STATE
    c, w = engine.resolve(want_candidates=True)
    _same(c, pc, "resolve after scenarios: candidates")
    _same(w, pw, "resolve after scenarios: winners")
    assert engine.last_device_ms > 0


def test_token_update_rebuilds_tables(engine, oracle_mod):
    fleet = scenario_fleets()["plain"]
    rows = scenario_rows(fleet.srv_arrival_rpm, 4)
    engine.upload(fleet)
    engine.resolve_scenarios(rows)
    out_tok = (fleet.srv_out_tokens // 2 + 7).astype(np.int32)
    engine.update_load(out_tokens=out_tok)
    cand, win = engine.resolve_scenarios(rows, want_candidates=True)
    f2 = fleet.take_servers(np.arange(fleet.n_servers))
    f2.srv_out_tokens[:] = out_tok
    for l, row in enumerate(rows):
        co, wo = oracle_mod.solve(with_arrival(f2, row))
        c, w = _blocks(fleet, cand, win, l)
        assert_allocs_equal(c, co, f"row {l} candidates after the token update")
        assert_allocs_equal(w, wo, f"row {l} winners after the token update")


def test_candidate_list_follows_loaded_servers(engine, oracle_mod):
    """The cached candidate list is rebuilt when a server idle in every row of one call carries load in the next."""
    fleet = scenario_fleets()["plain"]
    rows = scenario_rows(fleet.srv_arrival_rpm, 3)
    idle = rows.copy()
    idle[:, :5] = 0.0
    engine.upload(fleet)
    calls = [(r, engine.resolve_scenarios(r, want_candidates=True)) for r in (idle, rows, idle)]
    for k, (r, (cand, win)) in enumerate(calls):
        for l, row in enumerate(r):
            co, wo = oracle_mod.solve(with_arrival(fleet, row))
            c, w = _blocks(fleet, cand, win, l)
            assert_allocs_equal(c, co, f"call {k} row {l}: candidates")
            assert_allocs_equal(w, wo, f"call {k} row {l}: winners")


def test_bad_arguments(engine):
    L = engine._L
    fleet = scenario_fleets()["plain"]
    engine.upload(fleet)
    rows = scenario_rows(fleet.srv_arrival_rpm, 2)
    win = _abi.Allocs(2 * fleet.n_servers)
    wc = win.as_c()
    assert L.wva_resolve_scenarios(engine._h, 0, _abi.ptr(rows), None, C.byref(wc)) == _abi.WVA_ERR_BAD_ARG
    assert L.wva_resolve_scenarios(engine._h, -1, _abi.ptr(rows), None, C.byref(wc)) == _abi.WVA_ERR_BAD_ARG
    assert L.wva_resolve_scenarios(engine._h, 2, None, None, C.byref(wc)) == _abi.WVA_ERR_BAD_ARG
    assert L.wva_resolve_scenarios(engine._h, 2, _abi.ptr(rows), None, None) == _abi.WVA_ERR_BAD_ARG
    assert L.wva_resolve_scenarios(engine._h, 65536, _abi.ptr(rows), None, C.byref(wc)) == _abi.WVA_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        engine.resolve_scenarios(rows[:, :-1])
    fresh = Engine(0)
    try:
        rc = L.wva_resolve_scenarios(fresh._h, 2, _abi.ptr(rows), None, C.byref(wc))
        assert rc == _abi.WVA_ERR_STATE
        big = synth_fleet(8200, 4, seed=1)  # 65535 * 32800 records do not fit the kernels' int32 index
        fresh.upload(big)
        assert L.wva_resolve_scenarios(fresh._h, 65535, _abi.ptr(rows), None, C.byref(wc)) == _abi.WVA_ERR_UNSUPPORTED
    finally:
        fresh.close()


def test_streaming_fleet_full_size(engine):
    """The configs[4] streaming fleet (100 k pairs), 8 scenarios, every block against update_load + resolve."""
    fleet = synth_fleet(12500, 8, seed=45, max_batch_choices=(4, 8, 16, 32, 64, 128, 256))
    base = fleet.srv_arrival_rpm
    rng = np.random.Generator(np.random.PCG64(8))
    rows = np.stack([base * np.float32(f) for f in (1.0, 0.5, 1.25, 2.0, 4.0)] +
                    [np.where(rng.random(base.size) < 0.2, np.float32(0), base),
                     (base * rng.uniform(0.5, 1.5, base.size)).astype(np.float32),
                     np.where(base == 0, np.float32(100), base)]).astype(np.float32)
    _check(engine, None, fleet, rows, "configs[4]", oracle=False)
