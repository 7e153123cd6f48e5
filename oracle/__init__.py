"""Python loader for the CPU oracle (TEST INFRASTRUCTURE ONLY).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package (see oracle/wva_oracle.h).  The
product package never imports it.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libwva_oracle.so")


def build(force: bool = False) -> str:
    """Compile oracle/wva_oracle.c with the Go/amd64-semantics flags (oracle/Makefile)."""
    src = os.path.join(_HERE, "wva_oracle.c")
    hdr = os.path.join(_HERE, "wva_oracle.h")
    stale = (not os.path.exists(_SO)) or any(
        os.path.exists(p) and os.path.getmtime(p) > os.path.getmtime(_SO) for p in (src, hdr))
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "-s", "-B"], check=True)
    return _SO


class Metrics(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("throughput", "avg_resp_time", "avg_wait_time", "avg_num_in_serv",
                                          "avg_prefill_time", "avg_token_time", "max_rate", "rho")]


class TargetPerf(C.Structure):
    _fields_ = [("ttft", C.c_float), ("itl", C.c_float), ("tps", C.c_float)]


class TargetRate(C.Structure):
    _fields_ = [("rate_ttft", C.c_float), ("rate_itl", C.c_float), ("rate_tps", C.c_float)]


class ModelStats(C.Structure):
    _fields_ = [("is_valid", C.c_int32)] + [(n, C.c_float) for n in (
        "lambda_", "mu", "rho", "avg_resp_time", "avg_wait_time", "avg_serv_time", "avg_num_in_system",
        "avg_queue_length", "throughput", "avg_num_in_servers")] + [("sum_p", C.c_double)]


class AllocRec(C.Structure):
    _fields_ = [("feasible", C.c_int32), ("acc", C.c_int32), ("replicas", C.c_int32), ("batch", C.c_int32),
                ("cost", C.c_float), ("value", C.c_float), ("itl", C.c_float), ("ttft", C.c_float),
                ("rho", C.c_float), ("max_rate", C.c_float)]


class CellRec(C.Structure):
    _fields_ = [("flags", C.c_uint8), ("ttft", C.c_float), ("itl", C.c_float), ("rho", C.c_float),
                ("throughput", C.c_float)]


ALLOC_DTYPE = np.dtype([("feasible", "<i4"), ("acc", "<i4"), ("replicas", "<i4"), ("batch", "<i4"),
                        ("cost", "<f4"), ("value", "<f4"), ("itl", "<f4"), ("ttft", "<f4"), ("rho", "<f4"),
                        ("max_rate", "<f4")])
CELL_DTYPE = np.dtype([("flags", "u1"), ("ttft", "<f4"), ("itl", "<f4"), ("rho", "<f4"), ("throughput", "<f4")],
                      align=True)
assert ALLOC_DTYPE.itemsize == C.sizeof(AllocRec) and CELL_DTYPE.itemsize == C.sizeof(CellRec)

TYPE_TOTAL_DTYPE = np.dtype([("present", "<i4"), ("limit", "<i4"), ("count", "<i8"), ("cost", "<f4")], align=True)
DIFF_DTYPE = np.dtype([("old_acc", "<i4"), ("new_acc", "<i4"), ("old_replicas", "<i4"), ("new_replicas", "<i4"),
                       ("cost_diff", "<f4")])

EVAL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_float, C.POINTER(C.c_float))

_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):  # a stale library is rebuilt by build(), not here: bench.py may run on a read-only tree
        build()
    L = C.CDLL(_SO)
    f, i, vp = C.c_float, C.c_int, C.c_void_p
    L.wvao_prefill_time.restype = f
    L.wvao_prefill_time.argtypes = [f, f, i, f]
    L.wvao_decode_time.restype = f
    L.wvao_decode_time.argtypes = [f, f, f]
    L.wvao_effective_concurrency.restype = f
    L.wvao_effective_concurrency.argtypes = [f, f, f, f, f, i, i, i]
    L.wvao_within_tolerance.restype = i
    L.wvao_within_tolerance.argtypes = [f, f, f]
    L.wvao_binary_search.restype = i
    L.wvao_binary_search.argtypes = [f, f, f, EVAL_FN, vp, C.POINTER(f), C.POINTER(i)]
    L.wvao_mm1k_new.restype = vp
    L.wvao_mm1k_new.argtypes = [i]
    L.wvao_mm1k_free.argtypes = [vp]
    L.wvao_mm1k_solve.argtypes = [vp, f, f, C.POINTER(ModelStats)]
    L.wvao_mm1k_probs.restype = C.POINTER(C.c_double)
    L.wvao_mm1k_probs.argtypes = [vp]
    L.wvao_go_pow_uint.restype = C.c_double
    L.wvao_go_pow_uint.argtypes = [C.c_double, C.c_int64]
    L.wvao_model_new_rates.restype = vp
    L.wvao_model_new_rates.argtypes = [i, C.POINTER(C.c_float), i]
    L.wvao_analyzer_new.restype = vp
    L.wvao_analyzer_new.argtypes = [i, i, f, f, f, f, i, i]
    L.wvao_analyzer_free.argtypes = [vp]
    L.wvao_analyzer_rate_range.argtypes = [vp, C.POINTER(f), C.POINTER(f)]
    L.wvao_analyzer_serv_rate.restype = C.POINTER(f)
    L.wvao_analyzer_serv_rate.argtypes = [vp]
    L.wvao_analyzer_probs.restype = C.POINTER(C.c_double)
    L.wvao_analyzer_probs.argtypes = [vp]
    L.wvao_analyzer_K.restype = i
    L.wvao_analyzer_K.argtypes = [vp]
    L.wvao_analyzer_solves.restype = C.c_int64
    L.wvao_analyzer_solves.argtypes = [vp]
    L.wvao_model_solve.argtypes = [vp, f, f, C.POINTER(ModelStats)]
    L.wvao_analyze.restype = i
    L.wvao_analyze.argtypes = [vp, f, C.POINTER(Metrics)]
    L.wvao_size.restype = i
    L.wvao_size.argtypes = [vp, C.POINTER(TargetPerf), C.POINTER(TargetRate), C.POINTER(Metrics),
                            C.POINTER(TargetPerf)]
    L.wvao_eval_ttft.restype = i
    L.wvao_eval_ttft.argtypes = [vp, f, C.POINTER(f)]
    L.wvao_eval_itl.restype = i
    L.wvao_eval_itl.argtypes = [vp, f, C.POINTER(f)]
    L.wvao_create_allocation.argtypes = [vp, i, i, C.POINTER(AllocRec)]
    L.wvao_transition_penalty.restype = f
    L.wvao_transition_penalty.argtypes = [f, i, i, f, i, i, f]
    L.wvao_calculate.argtypes = [vp, vp]
    L.wvao_last_solves.restype = C.c_int64
    L.wvao_last_states.restype = C.c_int64
    L.wvao_solve_unlimited.argtypes = [vp, vp, vp]
    L.wvao_solve_greedy.argtypes = [vp, vp, vp]
    L.wvao_solve.argtypes = [vp, vp, vp]
    L.wvao_allocate_by_type.argtypes = [vp, vp, vp]
    L.wvao_allocation_diffs.argtypes = [vp, vp, vp]
    L.wvao_grid_solve.argtypes = [vp, vp, vp, vp]
    L.wvao_grid_cells.argtypes = [vp, vp, C.c_int64, C.c_int64, vp]
    L.wvao_sweep.argtypes = [vp, i] + [vp] * 6
    _lib = L
    return L


def _st(x: ModelStats) -> dict:
    d = {n: getattr(x, n) for n, _ in ModelStats._fields_}
    d["lambda"] = d.pop("lambda_")
    return d


def _mt(x: Metrics) -> dict:
    return {n: getattr(x, n) for n, _ in Metrics._fields_}


class Analyzer:
    """analyzer.QueueAnalyzer (pkg/analyzer/queueanalyzer.go:14-21) over the C oracle."""

    def __init__(self, max_batch, max_queue, alpha, beta, gamma, delta, in_tokens, out_tokens):
        self._h = lib().wvao_analyzer_new(max_batch, max_queue, alpha, beta, gamma, delta, in_tokens, out_tokens)
        if not self._h:
            raise ValueError("invalid configuration / request size")
        self.max_batch, self.max_queue = max_batch, max_queue

    def __del__(self):
        if getattr(self, "_h", None):
            lib().wvao_analyzer_free(self._h)
            self._h = None

    @property
    def K(self):
        return lib().wvao_analyzer_K(self._h)

    @property
    def solves(self):
        return lib().wvao_analyzer_solves(self._h)

    def rate_range(self):
        a, b = C.c_float(), C.c_float()
        lib().wvao_analyzer_rate_range(self._h, C.byref(a), C.byref(b))
        return a.value, b.value

    def serv_rate(self):
        return np.ctypeslib.as_array(lib().wvao_analyzer_serv_rate(self._h), (self.max_batch,)).copy()

    def probs(self):
        return np.ctypeslib.as_array(lib().wvao_analyzer_probs(self._h), (self.K + 1,)).copy()

    def solve(self, lam, mu=1.0):
        st = ModelStats()
        lib().wvao_model_solve(self._h, lam, mu, C.byref(st))
        return _st(st)

    def analyze(self, rate):
        """Returns (err, metrics); err 0 = ok (queueanalyzer.go:134-174)."""
        m = Metrics()
        err = lib().wvao_analyze(self._h, rate, C.byref(m))
        return err, (_mt(m) if err == 0 else None)

    def size(self, ttft, itl, tps):
        """Returns (err, rates, metrics, achieved) (queueanalyzer.go:185-255)."""
        t, r, m, a = TargetPerf(ttft, itl, tps), TargetRate(), Metrics(), TargetPerf()
        err = lib().wvao_size(self._h, C.byref(t), C.byref(r), C.byref(m), C.byref(a))
        if err:
            return err, None, None, None
        return 0, {n: getattr(r, n) for n, _ in TargetRate._fields_}, _mt(m), {n: getattr(a, n) for n, _ in
                                                                             TargetPerf._fields_}

    def eval_ttft(self, x):
        y = C.c_float()
        return lib().wvao_eval_ttft(self._h, x, C.byref(y)), y.value

    def eval_itl(self, x):
        y = C.c_float()
        return lib().wvao_eval_itl(self._h, x, C.byref(y)), y.value


class StateDependentModel:
    """analyzer.NewMM1ModelStateDependent(K, servRate) on its own (mm1modelstatedependent.go:16-24)."""

    def __init__(self, K, serv_rate):
        r = np.ascontiguousarray(serv_rate, np.float32)
        self._h = lib().wvao_model_new_rates(int(K), r.ctypes.data_as(C.POINTER(C.c_float)), int(r.size))
        if not self._h:
            raise ValueError("invalid model")
        self.K = int(K)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().wvao_analyzer_free(self._h)
            self._h = None

    def solve(self, lam, mu=1.0):
        st = ModelStats()
        lib().wvao_model_solve(self._h, lam, mu, C.byref(st))
        return _st(st)

    def probs(self):
        return np.ctypeslib.as_array(lib().wvao_analyzer_probs(self._h), (self.K + 1,)).copy()


class MM1K:
    def __init__(self, K):
        self.K = K
        self._h = lib().wvao_mm1k_new(K)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().wvao_mm1k_free(self._h)
            self._h = None

    def solve(self, lam, mu):
        st = ModelStats()
        lib().wvao_mm1k_solve(self._h, lam, mu, C.byref(st))
        return _st(st)

    def probs(self):
        return np.ctypeslib.as_array(lib().wvao_mm1k_probs(self._h), (self.K + 1,)).copy()


def go_pow_uint(x: float, n: int) -> float:
    """math.Pow(x, float64(n)) for an integer n >= 0, as restated from the Go standard library."""
    return float(lib().wvao_go_pow_uint(float(x), int(n)))


def mm1k_solve(K, lam, mu) -> dict:
    """MM1KModel.Solve for arrays of (K, lambda, mu): dict of numpy columns (the oracle of wva_mm1k_solve)."""
    K = np.asarray(K, np.int32)
    lam = np.asarray(lam, np.float32)
    mu = np.asarray(mu, np.float32)
    names = ("rho", "avg_num_in_system", "throughput", "avg_resp_time", "avg_serv_time", "avg_wait_time",
             "avg_queue_length")
    out = {n: np.zeros(K.size, np.float32) for n in names}
    out["is_valid"] = np.zeros(K.size, np.uint8)
    out["sum_p"] = np.zeros(K.size, np.float64)
    for i in range(K.size):
        st = MM1K(int(K[i])).solve(float(lam[i]), float(mu[i]))
        out["is_valid"][i] = st["is_valid"]
        out["rho"][i] = st["rho"]
        if st["is_valid"]:
            for n in names[1:]:
                out[n][i] = st[n]
            out["sum_p"][i] = st["sum_p"]
    return out


def binary_search(xmin, xmax, ytarget, fn):
    """utils.go:26-70. fn(x) -> y or raises. Returns (err, xstar, ind)."""
    def cb(_ctx, x, yp):
        try:
            yp[0] = fn(x)
            return 0
        except Exception:
            return 1
    xs, ind = C.c_float(), C.c_int()
    err = lib().wvao_binary_search(xmin, xmax, ytarget, EVAL_FN(cb), None, C.byref(xs), C.byref(ind))
    return err, xs.value, ind.value


def create_allocation(fleet, s, a) -> dict:
    rec = AllocRec()
    fc = fleet.as_c()
    lib().wvao_create_allocation(C.addressof(fc), s, a, C.byref(rec))
    return {n: getattr(rec, n) for n, _ in AllocRec._fields_}


def calculate(fleet) -> np.ndarray:
    """Server.Calculate for every server -> structured array [S, A]."""
    out = np.zeros((fleet.n_servers, fleet.n_acc), ALLOC_DTYPE)
    fc = fleet.as_c()
    lib().wvao_calculate(C.addressof(fc), out.ctypes.data)
    return out


def solve(fleet, cand=None):
    """Calculate + Solver.Solve -> (candidates [S, A], winners [S])."""
    if cand is None:
        cand = calculate(fleet)
    cand = cand.copy()
    win = np.zeros(fleet.n_servers, ALLOC_DTYPE)
    fc = fleet.as_c()
    lib().wvao_solve(C.addressof(fc), cand.ctypes.data, win.ctypes.data)
    return cand, win


def allocate_by_type(fleet, winners) -> np.ndarray:
    """System.AllocateByType over a solution (structured winners [S]) -> structured array [T]."""
    assert TYPE_TOTAL_DTYPE.itemsize == 24
    out = np.zeros(fleet.n_types, TYPE_TOTAL_DTYPE)
    win = np.ascontiguousarray(winners)
    fc = fleet.as_c()
    lib().wvao_allocate_by_type(C.addressof(fc), win.ctypes.data, out.ctypes.data)
    return out


def allocation_diffs(fleet, winners) -> np.ndarray:
    """CreateAllocationDiff(current, solution) per server -> structured array [S]."""
    out = np.zeros(fleet.n_servers, DIFF_DTYPE)
    win = np.ascontiguousarray(winners)
    fc = fleet.as_c()
    lib().wvao_allocation_diffs(C.addressof(fc), win.ctypes.data, out.ctypes.data)
    return out


def grid_solve(fleet, grid, want_cells=True):
    n = fleet.n_servers * fleet.n_acc * grid.batch.size * grid.replicas.size
    cells = np.zeros(n, CELL_DTYPE) if want_cells else None
    win = np.zeros(fleet.n_servers, ALLOC_DTYPE)
    fc, gc = fleet.as_c(), grid.as_c()
    lib().wvao_grid_solve(C.addressof(fc), C.addressof(gc), cells.ctypes.data if want_cells else None,
                          win.ctypes.data)
    return cells, win


def grid_cells(fleet, grid, c0, c1):
    cells = np.zeros(c1 - c0, CELL_DTYPE)
    fc, gc = fleet.as_c(), grid.as_c()
    lib().wvao_grid_cells(C.addressof(fc), C.addressof(gc), c0, c1, cells.ctypes.data)
    return cells


def sweep(fleet, n_rates):
    n = fleet.n_servers * fleet.n_acc * n_rates
    out = {"valid": np.zeros(n, np.uint8)}
    for k in ("rate", "ttft", "itl", "throughput", "rho"):
        out[k] = np.zeros(n, np.float32)
    fc = fleet.as_c()
    lib().wvao_sweep(C.addressof(fc), n_rates, *[out[k].ctypes.data for k in
                                                  ("valid", "rate", "ttft", "itl", "throughput", "rho")])
    return out


def last_counters():
    return lib().wvao_last_solves(), lib().wvao_last_states()
