"""Host-side mirror of the reference's optimizer interface over the C ABI.

``Engine`` plays the role of ``core.System`` + ``manager.Manager`` +
``solver.Optimizer`` for the hot path (pkg/manager/manager.go:13-27,
pkg/solver/optimizer.go:24-35, pkg/core/system.go:303-319): hand it the fleet
(``config.SystemSpec`` packed as a :class:`Fleet`), get candidate allocations
(``Server.Calculate``) and the per-server solution (``GenerateSolution``).  All compute
happens in the CUDA library; nothing here touches the oracle.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _abi, _lib
from ._abi import Allocs
from .fleet import Fleet, Grid


class WvaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"wva error {code}: {msg}")
        self.code = code


def greedy_solve(fleet: Fleet, candidates: Allocs):
    """``Solver.SolveGreedy`` + best-effort policies (pkg/solver/greedy.go:35-341) over a candidate table the
    caller already holds (``wva_solve_greedy``: host only, no GPU).  ``candidates`` [S * A] carries
    ``value`` = transition penalty (what ``Engine.analyze`` returns); it is modified in place where the reference
    scales best-effort allocations.  Returns (candidates, winners [S])."""
    L = _lib.lib()
    if candidates.n != fleet.n_servers * fleet.n_acc:
        raise ValueError("candidates must hold n_servers * n_acc records")
    win = Allocs(fleet.n_servers)
    fc, cc, wc = fleet.as_c(), candidates.as_c(), win.as_c()
    rc = L.wva_solve_greedy(C.byref(fc), C.byref(cc), C.byref(wc))
    if rc != 0:
        raise WvaError(rc, L.wva_strerror(rc).decode())
    return candidates, win


class Engine:
    """One engine per GPU (one process per GPU in multi-GPU runs)."""

    def __init__(self, device: int = 0):
        self._L = _lib.lib()
        h = C.c_void_p()
        rc = self._L.wva_create(C.byref(h), device)
        if rc != 0:
            raise WvaError(rc, self._L.wva_strerror(rc).decode() + " (the CUDA path has no CPU fallback)")
        self._h = h
        self._n_servers = self._n_acc = None  # shape of the fleet resident on the device

    def close(self):
        if getattr(self, "_h", None):
            self._L.wva_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise WvaError(rc, f"{self._L.wva_strerror(rc).decode()}: {self._L.wva_last_error(self._h).decode()}")

    # -- reference-shaped calls --------------------------------------------
    def analyze(self, fleet: Fleet) -> Allocs:
        """``Server.Calculate`` for every server -> candidates [S*A] (pkg/core/server.go:55-67)."""
        cand = Allocs(fleet.n_servers * fleet.n_acc)
        fc, cc = fleet.as_c(), cand.as_c()
        self._resident(fleet)
        self._check(self._L.wva_analyze(self._h, C.byref(fc), C.byref(cc)))
        return cand

    def solve(self, fleet: Fleet, want_candidates: bool = True):
        """``Manager.Optimize`` + ``GenerateSolution`` -> (candidates [S*A] | None, winners [S])."""
        cand = Allocs(fleet.n_servers * fleet.n_acc) if want_candidates else None
        win = Allocs(fleet.n_servers)
        fc, wc = fleet.as_c(), win.as_c()
        cc = cand.as_c() if cand is not None else None
        self._resident(fleet)
        self._check(self._L.wva_solve(self._h, C.byref(fc), C.byref(cc) if cc is not None else None, C.byref(wc)))
        return cand, win

    def grid_solve(self, fleet: Fleet, grid: Grid, want_cells: bool = False, out: Allocs | None = None):
        """Full (server x acc x batch x replica) grid -> (cells | None, winners [S]).

        ``out``: an ``Allocs`` of ``fleet.n_servers`` records to write the winners into (a reconcile
        loop reuses one instead of allocating ten columns per call)."""
        n = fleet.n_servers * fleet.n_acc * int(grid.batch.size) * int(grid.replicas.size)
        if out is not None and out.n != fleet.n_servers:
            raise ValueError("out must hold fleet.n_servers records")
        win = out if out is not None else Allocs(fleet.n_servers)
        cells = None
        cc = None
        if want_cells:
            cells = {"flags": np.zeros(n, np.uint8)}
            for k in ("ttft", "itl", "rho", "throughput"):
                cells[k] = np.zeros(n, np.float32)
            cc = _abi.CellsC(*[_abi.ptr(cells[k]) for k in ("flags", "ttft", "itl", "rho", "throughput")])
        fc, gc, wc = fleet.as_c(), grid.as_c(), win.as_c()
        self._resident(fleet)
        self._check(self._L.wva_grid_solve(self._h, C.byref(fc), C.byref(gc), C.byref(cc) if cc is not None else None,
                                           C.byref(wc)))
        return cells, win

    def sweep(self, fleet: Fleet, n_rates: int) -> dict:
        n = fleet.n_servers * fleet.n_acc * n_rates
        out = {"valid": np.zeros(n, np.uint8)}
        for k in ("rate", "ttft", "itl", "throughput", "rho"):
            out[k] = np.zeros(n, np.float32)
        oc = _abi.SweepOutC(*[_abi.ptr(out[k]) for k in ("valid", "rate", "ttft", "itl", "throughput", "rho")])
        fc = fleet.as_c()
        self._resident(fleet)
        self._check(self._L.wva_sweep(self._h, C.byref(fc), n_rates, C.byref(oc)))
        return out

    # -- streaming reconcile ------------------------------------------------
    def _resident(self, fleet: Fleet):
        """Every call that takes a fleet makes it the handle's resident fleet (the C side re-uploads it);
        ``resolve`` / ``update_load`` size their buffers from these counts, not from an older upload."""
        self._n_servers, self._n_acc = fleet.n_servers, fleet.n_acc

    def upload(self, fleet: Fleet):
        fc = fleet.as_c()
        self._check(self._L.wva_upload(self._h, C.byref(fc)))
        self._resident(fleet)

    def update_load(self, arrival_rpm=None, in_tokens=None, out_tokens=None):
        if self._n_servers is None:
            raise WvaError(_abi.WVA_ERR_STATE, "no resident fleet (call upload or a solve first)")
        a = np.ascontiguousarray(arrival_rpm, np.float32) if arrival_rpm is not None else None
        i = np.ascontiguousarray(in_tokens, np.int32) if in_tokens is not None else None
        o = np.ascontiguousarray(out_tokens, np.int32) if out_tokens is not None else None
        for name, col in (("arrival_rpm", a), ("in_tokens", i), ("out_tokens", o)):
            if col is not None and col.shape != (self._n_servers,):  # the C side copies exactly S entries
                raise ValueError(f"{name} must have {self._n_servers} entries (one per resident server), "
                                 f"got shape {col.shape}")
        self._check(self._L.wva_update_load(self._h, _abi.ptr(a) if a is not None else None,
                                            _abi.ptr(i) if i is not None else None,
                                            _abi.ptr(o) if o is not None else None))

    def resolve(self, want_candidates: bool = False):
        if self._n_servers is None:
            raise WvaError(_abi.WVA_ERR_STATE, "no resident fleet (call upload or a solve first)")
        cand = Allocs(self._n_servers * self._n_acc) if want_candidates else None
        win = Allocs(self._n_servers)
        wc = win.as_c()
        cc = cand.as_c() if cand is not None else None
        self._check(self._L.wva_resolve(self._h, C.byref(cc) if cc is not None else None, C.byref(wc)))
        return cand, win

    def resolve_scenarios(self, arrival_rpm, want_candidates: bool = False):
        """``resolve`` of the resident fleet under L arrival-rate scenarios in one call (``wva_resolve_scenarios``).

        ``arrival_rpm`` is ``[L, S]``: row l is every server's arrival rate (req/min) in scenario l.  Returns
        (candidates [L*S*A] | None, winners [L*S]); scenario l's block (records l*S*A.. / l*S..) equals
        ``update_load(arrival_rpm=row l)`` + ``resolve()``.  The resident fleet keeps its own load columns."""
        if self._n_servers is None:
            raise WvaError(_abi.WVA_ERR_STATE, "no resident fleet (call upload or a solve first)")
        a = np.ascontiguousarray(arrival_rpm, np.float32)
        if a.ndim != 2 or a.shape[1] != self._n_servers:  # the C side reads exactly L * S entries
            raise ValueError(f"arrival_rpm must have shape [L, {self._n_servers}] (one row per scenario, one column "
                             f"per resident server), got shape {a.shape}")
        n_scen, S = a.shape
        cand = Allocs(n_scen * S * self._n_acc) if want_candidates else None
        win = Allocs(n_scen * S)
        wc = win.as_c()
        cc = cand.as_c() if cand is not None else None
        self._check(self._L.wva_resolve_scenarios(self._h, n_scen, _abi.ptr(a), C.byref(cc) if cc is not None else None,
                                                  C.byref(wc)))
        return cand, win

    def summarize(self, n_types: int) -> dict:
        """``System.AllocateByType`` (pkg/core/system.go:271-300) and ``CreateAllocationDiff`` per server
        (pkg/core/allocation.go:353-380) over the most recent solution of this engine.

        Returns ``{"by_type": {present,count,limit,cost} arrays [T], "diff": {old_acc,new_acc,old_replicas,
        new_replicas,cost} arrays [S]}``; accelerator ids use ``ACC_NONE`` for "" and ``ACC_ABSENT`` for
        "none"."""
        if self._n_servers is None:
            raise WvaError(_abi.WVA_ERR_STATE, "no resident fleet (solve first)")
        T, S = int(n_types), self._n_servers
        by_type = {"present": np.zeros(T, np.uint8), "count": np.zeros(T, np.int64), "limit": np.zeros(T, np.int32),
                   "cost": np.zeros(T, np.float32)}
        diff = {"old_acc": np.zeros(S, np.int32), "new_acc": np.zeros(S, np.int32),
                "old_replicas": np.zeros(S, np.int32), "new_replicas": np.zeros(S, np.int32),
                "cost": np.zeros(S, np.float32)}
        sc = _abi.SummaryC(_abi.ptr(by_type["present"]), _abi.ptr(by_type["count"]), _abi.ptr(by_type["limit"]),
                           _abi.ptr(by_type["cost"]), _abi.ptr(diff["old_acc"]), _abi.ptr(diff["new_acc"]),
                           _abi.ptr(diff["old_replicas"]), _abi.ptr(diff["new_replicas"]), _abi.ptr(diff["cost"]))
        self._check(self._L.wva_summarize(self._h, C.byref(sc)))
        return {"by_type": by_type, "diff": diff}

    def mm1k_solve(self, K, lam, mu) -> dict:
        """``MM1KModel.Solve`` (pkg/analyzer/mm1kmodel.go:19-92) for arrays of (K, lambda, mu) triples; returns the
        model statistics as numpy columns (``is_valid``, ``rho``, ``avg_num_in_system``, ``throughput``,
        ``avg_resp_time``, ``avg_serv_time``, ``avg_wait_time``, ``avg_queue_length``, ``sum_p``)."""
        K = np.ascontiguousarray(K, np.int32)
        lam = np.ascontiguousarray(lam, np.float32)
        mu = np.ascontiguousarray(mu, np.float32)
        if not (K.shape == lam.shape == mu.shape and K.ndim == 1):
            raise ValueError("K, lam, mu must be 1-D arrays of one length")
        n = K.size
        out = {"is_valid": np.zeros(n, np.uint8)}
        names = ("rho", "avg_num_in_system", "throughput", "avg_resp_time", "avg_serv_time", "avg_wait_time",
                 "avg_queue_length")
        for name in names:
            out[name] = np.zeros(n, np.float32)
        out["sum_p"] = np.zeros(n, np.float64)
        oc = _abi.Mm1kOutC(_abi.ptr(out["is_valid"]), *[_abi.ptr(out[name]) for name in names], _abi.ptr(out["sum_p"]))
        self._check(self._L.wva_mm1k_solve(self._h, n, _abi.ptr(K), _abi.ptr(lam), _abi.ptr(mu), C.byref(oc)))
        return out

    # -- device-resident variants (multi-GPU driver, bench) -------------------
    def grid_solve_device(self, grid: Grid, winners_dev: _abi.AllocsC):
        gc = grid.as_c()
        self._check(self._L.wva_grid_solve_device(self._h, C.byref(gc), C.byref(winners_dev)))

    def resolve_device(self, winners_dev: _abi.AllocsC):
        self._check(self._L.wva_resolve_device(self._h, C.byref(winners_dev)))

    def synchronize(self):
        self._check(self._L.wva_synchronize(self._h))

    @property
    def stream(self) -> int:
        return int(self._L.wva_stream(self._h) or 0)

    @property
    def launch_count(self) -> int:
        return int(self._L.wva_launch_count(self._h))

    @property
    def last_kernel_ms(self) -> float:
        return float(self._L.wva_last_kernel_ms(self._h))

    @property
    def last_device_ms(self) -> float:
        return float(self._L.wva_last_device_ms(self._h))
