"""Fleets and arrival-rate scenario rows shared by the scenario tests (wva_resolve_scenarios)."""
import numpy as np

from workload_variant_autoscaler_b200 import synth_fleet

F32_SUBNORMAL = np.float32(1e-40)


def scenario_fleets():
    """Fleets covering every gate CreateAllocation has: keepAccelerator, zero-load servers, minReplicas = 0, TPS
    targets, missing profiles and targets, unknown models, batch sizes down to 1 and batch sizes from the profile."""
    plain = synth_fleet(12, 4, seed=5, max_batch_choices=(4, 8, 16, 32, 64))
    keep = synth_fleet(16, 3, seed=7, keep_accelerator=True, zero_load_frac=0.3, tps_frac=0.4,
                       max_batch_choices=(1, 2, 4, 8))
    gaps = synth_fleet(14, 3, seed=11, max_batch_choices=(1, 4, 16, 64), server_batch=False, tps_frac=0.3)
    gaps.srv_min_replicas[::3] = 0
    gaps.perf_present[0, 1] = 0     # no profile for (model 0, acc 1)
    gaps.perf_present[5, :] = 0     # model 5 has no profile at all
    gaps.srv_has_target[2] = 0      # no service-class target
    gaps.srv_model[4] = -1          # unknown model name
    gaps.srv_cur_acc[6] = -2        # current accelerator not in the table
    return {"plain": plain, "keep": keep, "gaps": gaps}


def scenario_rows(base, n_rows=None, *, seed=0):
    """Rows of arrival rates (req/min) derived from the base column: scaled, all zero, -0.0, negative, tiny,
    subnormal, huge and infinite, and a row that mixes these per server.  n_rows picks a prefix (1 = the base)."""
    base = np.asarray(base, np.float32)
    S = base.size
    rng = np.random.Generator(np.random.PCG64(seed))
    edge = np.array([0.0, -0.0, -3.0, 1e-30, F32_SUBNORMAL, 1e15, 1e30, np.inf], np.float32)
    rows = [base, base * np.float32(0.5), base * np.float32(2), base * np.float32(10), np.zeros(S, np.float32),
            np.full(S, -0.0, np.float32), -base - np.float32(1), np.full(S, 1e-30, np.float32),
            np.full(S, F32_SUBNORMAL, np.float32), np.full(S, 1e15, np.float32), np.full(S, 1e30, np.float32),
            np.full(S, np.inf, np.float32), np.where(rng.random(S) < 0.5, edge[rng.integers(0, edge.size, S)], base),
            base * np.float32(0.25), base * np.float32(3), base * np.float32(17),
            np.where(rng.random(S) < 0.3, np.float32(0), base * np.float32(1.5))]
    out = np.stack([np.asarray(r, np.float32) for r in rows])
    return out if n_rows is None else out[:n_rows]


def with_arrival(fleet, row):
    """A copy of the fleet with its arrival column replaced by one scenario row."""
    f = fleet.take_servers(np.arange(fleet.n_servers))
    f.srv_arrival_rpm[:] = np.asarray(row, np.float32)
    return f
