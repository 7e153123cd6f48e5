"""GPU: row resolution (DESIGN.md §3.2b) leaves the grid winners unchanged, bit for bit.

Without a cell table, grid_rows resolves the shared cells of a batch-invariant row into the row's smallest feasible
batch rank and grid_sort_local skips them.  The winners must equal those of the per-cell path (WVA_GRID_ROWRES=0),
of the path that writes the cell table (which never resolves), and of the CPU oracle.
"""
import ctypes as C
import zlib

import numpy as np
import pytest

from tests.test_gpu_parity import _adversarial_fleet
from tests.util import ALLOC_FIELDS, FLOAT_FIELDS, bits
from workload_variant_autoscaler_b200 import Grid, WvaError, config2_grid, synth_fleet

pytestmark = pytest.mark.gpu


def _column(w, name):
    return np.asarray(w[name] if isinstance(w, np.ndarray) else getattr(w, name))


def _assert_winners_equal(got, want, what, servers=None):
    """Every winner column of `got` (engine Allocs) equals `want` (Allocs or oracle records), floats as bits."""
    for name in ALLOC_FIELDS:
        g = _column(got, name)
        if servers is not None:
            g = g[servers]
        w = _column(want, name)
        if name in FLOAT_FIELDS:
            g, w = bits(g), bits(w)
        else:
            g, w = g.astype(np.int64), w.astype(np.int64)
        bad = np.nonzero(g != w)[0]
        assert bad.size == 0, f"{what}: winner {name} differs at servers {bad[:8].tolist()}: {g[bad[:4]]} vs {w[bad[:4]]}"


def _solve(engine, monkeypatch, fleet, grid, rowres, want_cells=False):
    monkeypatch.setenv("WVA_GRID_ROWRES", "1" if rowres else "0")
    _, win = engine.grid_solve(fleet, grid, want_cells=want_cells)
    return win


def _rows_resolved(engine):
    """Rows of the last grid solve that grid_rows resolved (diagnostic export of the library)."""
    L = engine._L
    L.wva_dbg_read_rows.restype = C.c_longlong
    L.wva_dbg_read_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
    cap = 1 << 22
    row_j = np.zeros(cap, np.int32)
    res = np.zeros(cap, np.uint8)
    n = L.wva_dbg_read_rows(engine._h, row_j.ctypes.data, res.ctypes.data, cap)
    return int(res[:n].sum())


def _check_three_ways(engine, monkeypatch, fleet, grid, what):
    """ROWRES on vs off vs the cell-table path; returns (winners, rows resolved), or (None, 0) when all three
    report the same error."""
    try:
        on = _solve(engine, monkeypatch, fleet, grid, True)
    except WvaError as exc:
        for rowres, want_cells in ((False, False), (True, True)):
            with pytest.raises(WvaError) as other:
                _solve(engine, monkeypatch, fleet, grid, rowres, want_cells)
            assert other.value.code == exc.code, what
        return None, 0
    n_res = _rows_resolved(engine)
    off = _solve(engine, monkeypatch, fleet, grid, False)
    assert _rows_resolved(engine) == 0
    cells = _solve(engine, monkeypatch, fleet, grid, True, want_cells=True)
    assert _rows_resolved(engine) == 0
    _assert_winners_equal(on, off, f"{what}: row resolution vs WVA_GRID_ROWRES=0")
    _assert_winners_equal(on, cells, f"{what}: row resolution vs the cell-table path")
    return on, n_res


@pytest.mark.parametrize("seed", range(42, 50))
def test_config2_fleets(engine, oracle_mod, monkeypatch, seed):
    fleet = synth_fleet(100, 4, seed=seed)
    grid = config2_grid()
    win, n_res = _check_three_ways(engine, monkeypatch, fleet, grid, f"seed {seed}")
    assert n_res > 0, "the configuration must exercise resolved rows"
    assert win.feasible.sum() > 50
    servers = np.random.default_rng(seed).choice(fleet.n_servers, 3, replace=False)
    _, win_o = oracle_mod.grid_solve(fleet.take_servers(servers), grid, want_cells=False)
    _assert_winners_equal(win, win_o, f"seed {seed}: against the oracle", servers=servers)


_BATCH = [1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48, 64, 96, 128, 200]


def _targeted(case):
    rng = np.random.default_rng(zlib.crc32(case.encode()))
    fleet = synth_fleet(24, 3, seed=77, tps_frac=0.3)
    grid = Grid(_BATCH, np.arange(1, 21))
    M, A = fleet.perf_beta.shape
    finite = True
    if case == "beta_delta_signs":
        # negative, zero and negative-zero coefficients, small enough that the service rates stay positive
        fleet.perf_gamma[:] = np.maximum(fleet.perf_gamma, 1.0)
        for col in (fleet.perf_beta, fleet.perf_delta):
            pick = rng.integers(0, 4, (M, A))
            col[pick == 0] = -1e-4
            col[pick == 1] = 0.0
            col[pick == 2] = -0.0
    elif case == "beta_delta_nonfinite":
        finite = False
        for col in (fleet.perf_beta, fleet.perf_delta):
            pick = rng.integers(0, 6, (M, A))
            col[pick == 0] = np.nan
            col[pick == 1] = np.inf
            col[pick == 2] = -np.inf
    elif case == "zero_slos":
        fleet.srv_slo_itl[::2] = 0.0
        fleet.srv_slo_ttft[1::2] = 0.0
        fleet.srv_slo_itl[::5] = 0.0
        fleet.srv_slo_ttft[::5] = 0.0
    elif case == "tps_everywhere":
        fleet.srv_slo_tps[:] = rng.choice([50.0, 500.0, 2000.0, 20000.0], fleet.n_servers)
    elif case == "min_replicas":
        fleet.srv_min_replicas[:] = rng.integers(2, 12, fleet.n_servers)
    elif case == "high_load":
        # rates above the stability limit of the small batch sizes at low replica levels
        fleet.srv_arrival_rpm[:] = np.exp(rng.uniform(np.log(2e4), np.log(5e5), fleet.n_servers))
        fleet.srv_slo_tps[::3] = 20000.0
    elif case == "unsorted_duplicates":
        grid = Grid([64, 3, 16, 16, 1, 128, 8, 3, 40, 200, 64, 2], np.arange(1, 21))
    elif case == "many_replicas":
        grid = Grid([1, 4, 16, 40, 64, 128, 256], np.arange(1, 100))
    return fleet, grid, finite


@pytest.mark.parametrize("case", ["beta_delta_signs", "beta_delta_nonfinite", "zero_slos", "tps_everywhere",
                                  "min_replicas", "high_load", "unsorted_duplicates", "many_replicas"])
def test_targeted_fleets(engine, oracle_mod, monkeypatch, case):
    fleet, grid, finite = _targeted(case)
    win, n_res = _check_three_ways(engine, monkeypatch, fleet, grid, case)
    if case in ("zero_slos", "tps_everywhere", "min_replicas", "unsorted_duplicates", "many_replicas"):
        assert n_res > 0, "the case must exercise resolved rows"
    if finite:
        assert win is not None, case
        _, win_o = oracle_mod.grid_solve(fleet, grid, want_cells=False)
        _assert_winners_equal(win, win_o, f"{case}: against the oracle")


def test_adversarial_fleets(engine, oracle_mod, monkeypatch):
    rng = np.random.default_rng(535353)
    resolved = 0
    for case in range(60):
        fleet = _adversarial_fleet(rng, case)
        grid = Grid(rng.integers(1, 60, int(rng.integers(1, 12))), rng.integers(1, 90, int(rng.integers(1, 24))))
        win, n_res = _check_three_ways(engine, monkeypatch, fleet, grid, f"adversarial case {case}")
        assert win is not None, case
        resolved += n_res
        _, win_o = oracle_mod.grid_solve(fleet, grid, want_cells=False)
        _assert_winners_equal(win, win_o, f"adversarial case {case}: against the oracle")
    assert resolved > 0
