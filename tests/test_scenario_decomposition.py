"""CPU: the decomposition wva_resolve_scenarios relies on (DESIGN §3.8), pinned on the oracle.

CreateAllocation under load is QueueAnalyzer.Size (which never reads the arrival rate) followed by a few per-load
steps and one final Analyze.  So every scenario's candidate can be computed from ONE Size per pair: the per-load
steps in float32 / float64 with Go's int(float64), then Analyze at the scenario's rate on the same analyzer, whose
previous solve belongs to another scenario.  This must equal oracle.create_allocation on the fleet with that
scenario's arrival column, bit for bit, for every scenario row, edge values included.
"""
import numpy as np
import pytest

from tests.scenarios import scenario_fleets, scenario_rows, with_arrival
from tests.util import bits

F32 = np.float32
I64_MIN = -(1 << 63)


def go_int(x: float) -> int:
    """int(float64) as Go compiles it for amd64 (CVTTSD2SQ): NaN and out-of-range values give the minimum int64."""
    if not np.isfinite(x) or not (-2.0 ** 63 <= x < 2.0 ** 63):
        return I64_MIN
    return int(x)


def i64_to_f32(v: int) -> np.float32:
    return np.array([v], np.int64).astype(np.float32)[0]  # one rounding, as float32(int64) in Go


def rate_free_gates(f, s, a):
    if f.srv_keep_acc[s] and f.srv_cur_acc[s] != -1 and f.srv_cur_acc[s] != a:
        return False
    if f.srv_in_tokens[s] < 0 or f.srv_out_tokens[s] < 0:
        return False
    m = int(f.srv_model[s])
    return 0 <= m < f.n_models and bool(f.perf_present[m, a]) and bool(f.srv_has_target[s])


def pair_batch(f, s, a):
    if f.srv_max_batch[s] > 0:
        return int(f.srv_max_batch[s])
    m = int(f.srv_model[s])
    return max(int(f.perf_max_batch[m, a]) * int(f.perf_at_tokens[m, a]) // int(f.srv_out_tokens[s]), 1)


def sized(oracle_mod, f, s, a):
    """(analyzer, rateStar) of one Size per pair, or (None, None) when Size or the analyzer is nil."""
    m, N = int(f.srv_model[s]), pair_batch(f, s, a)
    try:
        qa = oracle_mod.Analyzer(N, N * int(f.max_queue_to_batch_ratio), float(f.perf_alpha[m, a]),
                                 float(f.perf_beta[m, a]), float(f.perf_gamma[m, a]), float(f.perf_delta[m, a]),
                                 int(f.srv_in_tokens[s]), int(f.srv_out_tokens[s]))
    except ValueError:
        return None, None
    err, _, metrics, _ = qa.size(float(f.srv_slo_ttft[s]), float(f.srv_slo_itl[s]), float(f.srv_slo_tps[s]))
    return (qa, F32(metrics["throughput"])) if err == 0 else (qa, None)


def per_load(f, s, a, rpm, qa, rate_star):
    """allocation.go:134-163 at arrival rate rpm, from rateStar: the record create_allocation returns."""
    nil = dict(feasible=0, acc=-1, replicas=0, batch=0, cost=0.0, value=0.0, itl=0.0, ttft=0.0, rho=0.0, max_rate=0.0)
    m = int(f.srv_model[s])
    tps, K = F32(f.srv_slo_tps[s]), int(f.srv_out_tokens[s])
    total_rate = F32(rpm) / F32(60) if tps == 0 else tps / F32(K)
    nrep = max(go_int(np.ceil(np.float64(total_rate) / np.float64(rate_star))), int(f.srv_min_replicas[s]))
    inst = max(int(f.perf_acc_count[m, a]), 1)
    total = int((np.array([inst], np.int64) * np.array([nrep], np.int64))[0])  # wraps like Go's int64
    cost = F32(f.acc_cost[a]) * i64_to_f32(total)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        rate = total_rate / i64_to_f32(nrep)  # nrep = 0 (minReplicas 0, total rate 0) divides by zero, as in Go
    err, mt = qa.analyze(float(rate))
    if err != 0:
        return nil
    return dict(feasible=1, acc=a, replicas=int(np.int64(nrep).astype(np.int32)), batch=qa.max_batch, cost=cost,
                value=cost, itl=F32(mt["avg_token_time"]), ttft=F32(F32(mt["avg_wait_time"]) + F32(mt["avg_prefill_time"])),
                rho=F32(mt["rho"]), max_rate=rate_star / F32(1000))


def assert_rec_equal(got, want, what):
    for k in ("feasible", "acc", "replicas", "batch"):
        assert int(got[k]) == int(want[k]), f"{what}: {k} got {got[k]} want {want[k]}"
    for k in ("cost", "value", "itl", "ttft", "rho", "max_rate"):
        assert bits([got[k]])[0] == bits([want[k]])[0], f"{what}: {k} got {got[k]!r} want {want[k]!r}"


@pytest.mark.parametrize("name", ["plain", "keep", "gaps"])
def test_size_once_then_per_load_steps(oracle_mod, name):
    fleet = scenario_fleets()[name]
    rows = np.concatenate([scenario_rows(fleet.srv_arrival_rpm, seed=3),
                           np.full((1, fleet.n_servers), np.nan, np.float32)])
    scen = [with_arrival(fleet, r) for r in rows]
    n_load = 0
    for s in range(fleet.n_servers):
        for a in range(fleet.n_acc):
            if not rate_free_gates(fleet, s, a) or fleet.srv_out_tokens[s] <= 0:
                continue
            qa, rate_star = sized(oracle_mod, fleet, s, a)
            # the rows in a shuffled order: the analyzer's previous solve is some other scenario's final Analyze
            for l in np.random.Generator(np.random.PCG64(s * 31 + a)).permutation(len(rows)):
                rpm = F32(rows[l][s])
                if rpm == 0 or rpm < 0:
                    continue  # the zero-load and negative-rate gates: no Size at all
                want = oracle_mod.create_allocation(scen[l], s, a)
                if rate_star is None:
                    assert want["feasible"] == 0, f"{name} s{s} a{a} row {l}: Size is nil"
                    continue
                assert_rec_equal(per_load(fleet, s, a, rpm, qa, rate_star), want, f"{name} s{s} a{a} row {l} ({rpm})")
                n_load += 1
    assert n_load > 50


def test_rate_star_is_the_same_in_every_scenario(oracle_mod):
    """max_rate = rateStar / 1000 of every pair feasible in several scenarios is one value."""
    fleet = scenario_fleets()["plain"]
    rows = scenario_rows(fleet.srv_arrival_rpm)[[0, 1, 2, 3, 13, 14, 15]]
    seen = {}
    for r in rows:
        cand, _ = oracle_mod.solve(with_arrival(fleet, r))
        for i in np.nonzero(cand.reshape(-1)["feasible"])[0]:
            if cand.reshape(-1)["acc"][i] >= 0:
                seen.setdefault(int(i), set()).add(int(bits([cand.reshape(-1)["max_rate"][i]])[0]))
    assert len(seen) > 20 and all(len(v) == 1 for v in seen.values())
