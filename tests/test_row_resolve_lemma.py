"""CPU check of the lemma behind row resolution (DESIGN.md §3.2b).

On a batch-invariant row a shared cell depends on its batch size N only through eff = min(effu, N).  With alpha,
gamma, w0 and effu finite, beta >= 0 and d_in >= 0 (or no input tokens), the SLO part of the cell's feasibility is a
down-set in N: once it fails it fails for every larger N.  This is a float32 restatement of shared_cell_metrics_inv
and the SLO comparisons of cell_feasible (every operation rounds to nearest, as on the device), evaluated over random
operands that meet the preconditions, including overflow to +inf and SLOs placed one ulp around the metrics.
"""
import numpy as np

F32 = np.float32


def _slo_feasible(alpha, beta, gamma, d_in, in_zero, w0, effu, slo_itl, slo_ttft, n):
    """[rows, len(n)] SLO feasibility of shared_cell_metrics_inv + cell_feasible (replica and TPS terms are row
    constants or depend on the batch size alone, so they are left out)."""
    with np.errstate(over="ignore", invalid="ignore"):
        eff = np.minimum(effu[:, None], n[None, :].astype(F32))
        itl = alpha[:, None] + beta[:, None] * eff
        prefill = np.where(in_zero[:, None], F32(0), gamma[:, None] + d_in[:, None] * eff)
        ttft = w0[:, None] + prefill
        ok_itl = (slo_itl[:, None] == 0) | (itl <= slo_itl[:, None])
        ok_ttft = (slo_ttft[:, None] == 0) | (ttft <= slo_ttft[:, None])
    assert itl.dtype == F32 and ttft.dtype == F32
    return ok_itl & ok_ttft, itl, ttft


def _operands(rng, rows, beta_sign=1.0):
    def logu(lo, hi):
        return np.exp(rng.uniform(np.log(lo), np.log(hi), rows)).astype(F32)

    alpha = logu(1e-3, 1e3) * rng.choice([1, -1], rows).astype(F32)
    alpha[rng.random(rows) < 0.05] = F32(3e38)  # alpha + beta*eff overflows to +inf
    beta = (logu(1e-6, 1e3) * F32(beta_sign)).astype(F32)
    beta[rng.random(rows) < 0.1] = F32(0)
    beta[rng.random(rows) < 0.05] = F32(-0.0)
    beta[rng.random(rows) < 0.03] = F32(3e36 * beta_sign)
    gamma = logu(1e-3, 1e4)
    gamma[rng.random(rows) < 0.1] = F32(0)
    d_in = logu(1e-7, 1e3)
    d_in[rng.random(rows) < 0.1] = F32(0)
    in_zero = rng.random(rows) < 0.1
    w0 = logu(1e-6, 1e6)
    w0[rng.random(rows) < 0.2] = F32(0)
    effu = logu(1e-3, 5e3)
    effu[rng.random(rows) < 0.1] = F32(0)
    return alpha, beta, gamma, d_in, in_zero, w0, effu


def _slos_at_the_edges(rng, itl, ttft):
    """SLOs equal to a metric at a random batch size, one ulp either side, 0 (no target) or +inf."""
    rows, n = itl.shape
    pick = rng.integers(0, n, rows)
    out = []
    for m in (itl, ttft):
        slo = m[np.arange(rows), pick].copy()
        nudge = rng.integers(-1, 2, rows)
        slo = np.where(nudge < 0, np.nextafter(slo, F32(-np.inf)), np.where(nudge > 0, np.nextafter(slo, F32(np.inf)), slo))
        slo[rng.random(rows) < 0.1] = F32(0)
        slo[rng.random(rows) < 0.03] = F32(np.inf)
        out.append(slo.astype(F32))
    return out


def _is_down_set(feas):
    return ~np.any(np.diff(feas.astype(np.int8), axis=1) > 0, axis=1)


def test_shared_cell_feasibility_is_a_down_set_in_the_batch_size():
    rng = np.random.default_rng(20261017)
    n = np.arange(1, 2049)
    rows = 4000
    for _ in range(5):
        ops = _operands(rng, rows)
        inf_slo = np.full(rows, np.inf, F32)
        _, itl, ttft = _slo_feasible(*ops, inf_slo, inf_slo, n)
        slo_itl, slo_ttft = _slos_at_the_edges(rng, itl, ttft)
        feas, _, _ = _slo_feasible(*ops, slo_itl, slo_ttft, n)
        ok = _is_down_set(feas)
        assert ok.all(), f"{(~ok).sum()} rows are not a down-set; first: {[o[~ok][0] for o in ops]}"
        # the operands reach both outcomes, and rows that switch from feasible to infeasible
        assert feas.any() and (~feas).any()
        assert (feas[:, 0] & ~feas[:, -1]).sum() > rows // 20


def test_negative_beta_breaks_the_lemma():
    """The precondition beta >= 0 is needed: with beta < 0 the decode time falls as N grows, and rows that are
    infeasible at small N become feasible later (grid_rows leaves such rows to the per-cell path)."""
    rng = np.random.default_rng(7)
    n = np.arange(1, 2049)
    rows = 4000
    ops = _operands(rng, rows, beta_sign=-1.0)
    inf_slo = np.full(rows, np.inf, F32)
    _, itl, ttft = _slo_feasible(*ops, inf_slo, inf_slo, n)
    slo_itl, slo_ttft = _slos_at_the_edges(rng, itl, ttft)
    feas, _, _ = _slo_feasible(*ops, slo_itl, slo_ttft, n)
    assert not _is_down_set(feas).all()
