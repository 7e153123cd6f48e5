"""Edge fleets for the streaming solver's exponent windows, and a CPU check that they reach every band.

The solver's path for a state (reciprocal step, exact division, block of 4 or 16 unchecked steps, bail to the
stored-vector fallback) is chosen by exponent windows (DESIGN.md §3.1, §3.2).  The parity suites draw their fleets
from `synth_fleet`, whose chains stay far from the window edges, so a wrong bound would pass them.  The fleets below
are built to land on each edge; `test_edge_fleets_reach_every_band` proves with the band calculator (tests/bands.py,
the oracle's service rates, the entries' own float32 lambda formulas) that each band is hit by at least one solve of
the entry it targets, and tests/test_gpu_windows.py compares the device with the oracle on the same fleets.

Linear rates (alpha = 1, beta = gamma = delta = 0, no input tokens, two output tokens) give servRate[n-1] = n, so a
chain at lambda is p[n] = lambda^n / n!: its peak and sum are set by lambda and N alone.
"""
import math

import numpy as np
import pytest

import oracle
from tests.bands import chain_bands, f32, row_bands
from workload_variant_autoscaler_b200 import Grid, synth_fleet

# ---------------------------------------------------------------------------------------------------------------
# fleets
# ---------------------------------------------------------------------------------------------------------------
WIDE_N = (480, 600, 614, 615, 616, 620, 640, 720)   # size / resolve / sweep: peaks 2^686 .. 2^880 .. overflow
RAISED_N, RAISED_RATES = 1400, 2048                 # sweep indices 896..899: pass-2 raised band, peak below 2^880
RAISED_IDX = (896, 897, 898, 899)
NARROW_LAMBDA = (419.0, 420.0, 429.0, 429.5, 430.0, 431.0, 715.0)  # grid lambda at one replica
NARROW_BATCH = (420, 424, 432, 440, 720, 2048)
SHARP_N, SHARP_RATES = 96, 8000                     # sweep indices SHARP_IDX (one warp): a narrow peak over 2^880
SHARP_IDX = range(38 * 32, 39 * 32)


def _linear(n_servers, batch, rpm, *, alpha=1.0, slo_ttft=0.0, slo_itl=0.0):
    f = synth_fleet(n_servers, 1, seed=31, n_models=n_servers, zero_load_frac=0.0, tps_frac=0.0)
    f.perf_alpha[:] = alpha
    f.perf_beta[:] = 0.0
    f.perf_gamma[:] = 0.0
    f.perf_delta[:] = 0.0
    f.perf_acc_count[:] = 1
    f.srv_in_tokens[:] = 0
    f.srv_out_tokens[:] = 2
    f.srv_max_batch[:] = batch
    f.srv_arrival_rpm[:] = rpm
    f.srv_slo_tps[:] = 0.0
    f.srv_slo_ttft[:] = slo_ttft
    f.srv_slo_itl[:] = slo_itl
    f.srv_min_replicas[:] = 1
    f.srv_cur_acc[:] = -1
    f.srv_cur_replicas[:] = 0
    f.srv_cur_cost[:] = 0.0
    return f


def wide_fleet():
    """One server per N in WIDE_N: Size's searches start at RateRange.Max/1000, where the peak crosses 2^880 between
    N = 614 and 615 and the sum 2^900 between 620 and 640; N = 720 overflows (the reference rescales).  The TTFT target
    makes Size bisect, the ITL target is met everywhere (ITL = alpha)."""
    return _linear(len(WIDE_N), np.array(WIDE_N), 60.0 * 1000.0 * 200.0, slo_ttft=5.0, slo_itl=2.0)


def raised_fleet():
    """N = 1400 at one replica with lambda = 613 (Size's final Analyze; the sweep's indices RAISED_IDX come close to it):
    the chain peaks at 2^878 and ends (exact early termination) with a sum of 2^884, so
    pass 2 divides by the sum with its lower bound raised to 2^-76 and the states just above the termination
    threshold 2^-78 take div.rn.f64."""
    return _linear(1, np.array([RAISED_N]), 613.0 * 60000.0, slo_ttft=1e6, slo_itl=2.0)


def rate_edge_fleet():
    """N = 1, servRate[0] = 1/alpha, at both edges of the half-open window [2^-60, 2^60):
    servers 0, 1   servRate[0] at 2^60 (outside) and one float32 step below it (inside);
    servers 2, 3   servRate[0] at 2^-60 (inside) and one step below it (outside);
    servers 4, 5   the sweep's first lambda, RateRange.Min/1000, at 2^-60 (inside) and two steps below it (outside;
                   below 2^-60 the float32 steps halve, one step of alpha moves lambda by two);
    servers 6, 7   Size's lambda, RateRange.Max/1000, at 2^-60 (inside) and one step below it (outside)."""
    hi_a = np.float32(2.0 ** -60)
    lo_a = np.float32(2.0 ** 60)
    min_a = np.float32(1152921559367680.0)   # RateRange.Min/1000 = 2^-60 exactly
    max_a = np.float32(1151768597945647104.0)   # RateRange.Max/1000 = 2^-60 exactly
    up = np.float32(np.inf)
    f = _linear(8, np.ones(8, np.int64), 60.0 * 1e20, slo_ttft=0.0, slo_itl=0.0)
    f.perf_alpha[:, 0] = [hi_a, np.nextafter(hi_a, up), lo_a, np.nextafter(lo_a, up), min_a, np.nextafter(min_a, up),
                          max_a, np.nextafter(max_a, up)]
    return f


def sharp_peak_fleet():
    """N = 96 with a negative beta that brings the decode time of the last batch size close to 0: servRate rises from
    1 to 9e3 over the head and jumps to 3.9e5 at N.  At lambda ~ 6e4 the chain climbs 3-16 doublings per state to a
    peak just above 2^880 at state 95 and falls 2.7 doublings per state after it.  A 4-step block starting at state 93
    below 2^880 ends at 97 below it again; only the 3 e_hi margin of the 4-step window (e_hi = 16 here) stops the
    blocks early enough for the solver to see the peak and bail.  All 32 lanes of the warp that solves the sweep
    indices SHARP_IDX are in that situation, so the warp's block votes keep the blocks at states 1, 5, 9, ..."""
    f = _linear(1, np.array([SHARP_N]), 60.0 * 1000.0, slo_ttft=0.0, slo_itl=0.0)
    f.perf_beta[:] = np.float32(-(1 - 2.0 ** -12) / SHARP_N)
    return f


def narrow_fleet():
    """Grid servers at one-replica lambdas around the narrow instantiation's edges: cell peaks across 2^600
    (lambda 419 / 420), cell sums across 2^620 and row sums just below (429, 429.5) and at or above (430, 431) 2^620
    for the 2048-entry row chain; lambda 715 overflows at batch 720 and in the row."""
    rpm = np.array([lam * 60000.0 for lam in NARROW_LAMBDA], np.float32)
    return _linear(len(NARROW_LAMBDA), 1, rpm, slo_ttft=1e6, slo_itl=2.0)


def narrow_grid():
    return Grid(list(NARROW_BATCH), [1, 2])


def overflow_fleet():
    """test_gpu_parity's N = 1024 rescale fleet (two servers near saturation), for every entry including the sweep."""
    fleet = synth_fleet(2, 1, seed=29, max_batch_choices=(1024,))
    fleet.perf_alpha[:] = 7.47
    fleet.perf_beta[:] = 0.0001
    fleet.perf_gamma[:] = 1.0
    fleet.perf_delta[:] = 0.00001
    fleet.srv_in_tokens[:] = 64
    fleet.srv_out_tokens[:] = 64
    fleet.srv_slo_tps[:] = 0
    fleet.srv_slo_itl[:] = 0
    fleet.srv_slo_ttft[:] = 0
    fleet.srv_arrival_rpm[:] = [60.0 * 2100, 60.0 * 1900]
    return fleet


# ---------------------------------------------------------------------------------------------------------------
# the lambdas each entry evaluates, restated in float32
# ---------------------------------------------------------------------------------------------------------------
def _analyzer(fleet, s, N):
    m = int(fleet.srv_model[s])
    return oracle.Analyzer(int(N), int(N) * fleet.max_queue_to_batch_ratio, float(fleet.perf_alpha[m, 0]),
                           float(fleet.perf_beta[m, 0]), float(fleet.perf_gamma[m, 0]), float(fleet.perf_delta[m, 0]),
                           int(fleet.srv_in_tokens[s]), int(fleet.srv_out_tokens[s]))


def sweep_lambdas(rmin, rmax, n_rates):
    """sweep_kernel: rate_i = rmin + (rmax * 0.999 - rmin) * (i / (n - 1)), lambda = rate / 1000."""
    hi = f32(f32(rmax) * f32(0.999))
    span = f32(hi - f32(rmin))
    out = []
    for i in range(n_rates):
        frac = f32(f32(i) / f32(n_rates - 1)) if n_rates > 1 else f32(0)
        out.append(f32(f32(f32(rmin) + f32(span * frac)) / f32(1000)))
    return out


def size_lambdas(qa, slo_ttft):
    """Size (queueanalyzer.go:185-255): the TTFT search's evaluations, traced through the oracle's BinarySearch
    (RateRange.Max/1000 first), then the final Analyze."""
    rmin, rmax = qa.rate_range()
    lmin, lmax = f32(f32(rmin) / f32(1000)), f32(f32(rmax) / f32(1000))
    seen = []
    if slo_ttft > 0:
        def ev(x):
            seen.append(f32(x))
            err, y = qa.eval_ttft(x)
            if err:
                raise ValueError
            return y
        oracle.binary_search(float(lmin), float(lmax), float(slo_ttft), ev)
    return seen + [lmax]


def grid_lambda(fleet, s, r):
    total = f32(f32(fleet.srv_arrival_rpm[s]) / f32(60))
    return f32(f32(total / f32(r)) / f32(1000))


def solves_by_entry():
    """{entry: [(fleet name, N, K, lambda, serv_rate, extra)]} for the edge fleets."""
    out = {"size": [], "sweep": [], "grid": [], "row": []}
    for name, fleet in (("wide", wide_fleet()), ("raised", raised_fleet()), ("rate_edge", rate_edge_fleet()),
                        ("overflow", overflow_fleet()), ("sharp", sharp_peak_fleet())):
        for s in range(fleet.n_servers):
            N = int(fleet.srv_max_batch[s])
            qa = _analyzer(fleet, s, N)
            sr = qa.serv_rate()
            K = N + N * fleet.max_queue_to_batch_ratio
            for lam in size_lambdas(qa, float(fleet.srv_slo_ttft[s])):
                out["size"].append((name, N, K, lam, sr, None))
            rec = oracle.create_allocation(fleet, s, 0)   # CreateAllocation's last Analyze: total rate / replicas
            if rec["feasible"]:
                out["size"].append((name, N, K, grid_lambda(fleet, s, rec["replicas"]), sr, None))
            n_rates = {"raised": RAISED_RATES, "sharp": SHARP_RATES}.get(name, 64)
            lams = sweep_lambdas(*qa.rate_range(), n_rates)
            idx = {"raised": RAISED_IDX, "sharp": SHARP_IDX}.get(name, range(n_rates))
            for i in idx:
                out["sweep"].append((name, N, K, lams[i], sr, i))
    fleet, grid = narrow_fleet(), narrow_grid()
    bmax = int(max(grid.batch))
    for s in range(fleet.n_servers):
        sr = _analyzer(fleet, s, bmax).serv_rate()
        for r in grid.replicas:
            lam = grid_lambda(fleet, s, int(r))
            out["row"].append(("narrow", bmax, None, lam, sr, int(r)))
            for b in grid.batch:
                b = int(b)
                rmax = f32(f32(f32(sr[b - 1]) * f32(1 - f32(0.001))) * f32(1000))
                if f32(lam * f32(1000)) <= rmax:   # Analyze rejects rates above RateRange.Max
                    out["grid"].append(("narrow", b, b + b * fleet.max_queue_to_batch_ratio, lam, sr[:b], int(r)))
    return out


# ---------------------------------------------------------------------------------------------------------------
# bands
# ---------------------------------------------------------------------------------------------------------------
def _ulps_to(x, e):
    return abs(int(np.float32(x).view(np.int32)) - int(np.float32(2.0 ** e).view(np.int32)))


def _near_rate_edge(b, sr, N, e):
    return min(_ulps_to(v, e) for v in (b["lam"], sr[0], sr[N - 1])) <= 2


WIDE_BANDS = {
    "peak just below 2^880": lambda b: 876 <= b["e_peak"] < 880,
    "peak at or above 2^880 (bails)": lambda b: 880 <= b["e_peak"] < 1024,
    "sum approaching 2^900": lambda b: 894 <= b["e_sum"] < 900 and b["e_peak"] < 1024,
    "sum at or above 2^900 (bails)": lambda b: 900 <= b["e_sum"] < 1024,
    "raised pass-2 band non-empty, no bail": lambda b: b["n_raised"] > 0 and b["e_peak"] < 880 and b["e_sum"] < 900,
    "beyond 2^1024 (rescale)": lambda b: b["overflow"],
    "rate or lambda one float32 step below 2^60 (inside)": lambda b: b["rates_ok"] and b["near_hi"],
    "rate at 2^60 (outside)": lambda b: not b["rates_ok"] and b["near_hi"],
    "rate or lambda at 2^-60 (inside)": lambda b: b["rates_ok"] and b["near_lo"],
    "rate or lambda one float32 step below 2^-60 (outside)": lambda b: not b["rates_ok"] and b["near_lo"],
    "e_lo <= -20": lambda b: b["e_lo"] is not None and b["e_lo"] <= -20,
}
SWEEP_BANDS = {
    "4-step block could step over a peak above 2^880 (the 3 e_hi margin decides)":
        lambda b: b["block_straddle"] and b["e_hi"] > 0 and b["e_sum"] < 900,
}
NARROW_BANDS = {
    "cell peak just below 2^600": lambda b: 596 <= b["e_peak"] < 600,
    "cell peak at or above 2^600 (bails)": lambda b: 600 <= b["e_peak"] < 1024,
    "cell sum just below 2^620": lambda b: 616 <= b["e_sum"] < 620,
    "cell sum at or above 2^620": lambda b: 620 <= b["e_sum"] < 1024,
    "cell beyond 2^1024 (rescale)": lambda b: b["overflow"],
}
ROW_BANDS = {
    "row sum just below 2^620, shared": lambda b: b["shared"] and 616 <= b["e_sum"] < 620,
    "row sum at or above 2^620, not shared": lambda b: (not b["shared"]) and b.get("sum_ok") is False,
}

# Bands no input that Analyze accepts can reach, with the reason.  They stay listed so that a change to the windows
# or to the service-rate model that makes one reachable shows up here.
UNREACHABLE = {
    "grid: cell sum >= 2^616 with peak < 2^600": "as below, the sum is at most about 2^11 times the peak, so every "
    "narrow cell near the 2^620 sum bound has already left the 2^600 peak bound; the sum bound of the narrow "
    "instantiation never binds first (the row solve's does: row bands above)",
    "sum >= 2^900 with peak < 2^880": "the sum of a chain that ends by early termination or at K = 11N is at most about "
    "2^10 times its peak here (tail ratio lambda / servRate[N-1] <= 0.999, so the tail adds at most 1000 peaks, the "
    "head at most N): a peak below 2^880 keeps the sum below 2^900",
    "16-step blocks disabled on a WIDE entry": "they need 15 (max(e_hi, 0) - min(e_lo, 0)) >= 1159.  servRate[n-1] = "
    "n / (c0 + c1 n) in float32 varies by at most N 2^25 over the table, so e_hi - e_lo <= 47, and the size, resolve "
    "and sweep lambdas are >= RateRange.Min/1000 = servRate[0] / 1000, so -e_lo <= 57",
    "p below 2^-280 before termination": "servRate[n-1] = n / (c0 + c1 n) is monotone in n, so the chain is unimodal; "
    "p[1] >= 2^-120 (rates and lambda in [2^-60, 2^60)) puts the termination threshold 2^-78 min(1, p[1]) above "
    "2^-198, and a chain below it is past its mode with lambda at least 2^13 float32 steps below servRate[N-1]",
}


def _hits():
    solves = solves_by_entry()
    entries = (("size", WIDE_BANDS), ("sweep", {**WIDE_BANDS, **SWEEP_BANDS}), ("grid", NARROW_BANDS))
    hits = {f"{e}: {k}": 0 for e, bands in entries + (("row", ROW_BANDS),) for k in bands}
    for entry, bands in entries:
        cache = {}
        for (_name, N, K, lam, sr, _x) in solves[entry]:
            key = (N, K, float(lam), float(sr[0]))
            if key not in cache:
                b = chain_bands(sr, N, K, lam)
                b["near_hi"], b["near_lo"] = _near_rate_edge(b, sr, N, 60), _near_rate_edge(b, sr, N, -60)
                cache[key] = b
            for k, pred in bands.items():
                hits[f"{entry}: {k}"] += bool(pred(cache[key]))
    for (_name, L, _K, lam, sr, _r) in solves["row"]:
        b = row_bands(sr, L, lam)
        for k, pred in ROW_BANDS.items():
            hits[f"row: {k}"] += bool(pred(b))
    return hits


def test_edge_fleets_reach_every_band():
    hits = _hits()
    report = "\n".join(f"  {n:6d}  {k}" for k, n in hits.items())
    report += "\n  unreachable with inputs Analyze accepts:\n" + "\n".join(f"    {k}: {v}" for k, v in UNREACHABLE.items())
    missed = [k for k, n in hits.items() if n == 0]
    assert not missed, f"bands without a solve: {missed}\n{report}"


def test_band_calculator_matches_known_chains():
    """The calculator against hand-derived chains: p[n] = lambda^n / n! at N = 1400 (the raised band needs a sum above
    2^680), and the N = 615 chain of the wide fleet peaking at exactly 2^880."""
    sr = _analyzer(raised_fleet(), 0, RAISED_N).serv_rate()
    assert np.array_equal(sr, np.arange(1, RAISED_N + 1, dtype=np.float32))
    b = chain_bands(sr, RAISED_N, 11 * RAISED_N, f32(613.0))
    assert (b["e_peak"], b["e_sum"], b["n_raised"]) == (878, 884, 2)
    assert b["j_end"] < 11 * RAISED_N and not b["overflow"]
    # Stirling: log2(lambda^n / n!) at n = lambda is about lambda log2(e) - log2(2 pi lambda) / 2
    assert abs(b["e_peak"] - (613 * math.log2(math.e) - 0.5 * math.log2(2 * math.pi * 613))) < 1.5
    qa = _analyzer(wide_fleet(), WIDE_N.index(615), 615)
    lmax = f32(f32(qa.rate_range()[1]) / f32(1000))
    assert chain_bands(qa.serv_rate(), 615, 6765, lmax)["e_peak"] == 880


# ---------------------------------------------------------------------------------------------------------------
# the oracle against 200-bit arithmetic on the edge chains
# ---------------------------------------------------------------------------------------------------------------
def _mp_stats(sr, N, K, lam):
    mpmath = pytest.importorskip("mpmath")
    mpmath.mp.prec = 200
    lam_m = mpmath.mpf(float(lam))
    rates = [mpmath.mpf(float(x)) for x in sr[:N]]
    p = [mpmath.mpf(1)]
    for n in range(K):
        p.append(p[-1] * lam_m / rates[min(n, N - 1)])
    total = mpmath.fsum(p)
    in_sys = mpmath.fsum(i * p[i] for i in range(1, K + 1)) / total
    head = mpmath.fsum(p[: N + 1]) / total
    in_serv = mpmath.fsum(i * p[i] for i in range(1, N + 1)) / total + (1 - head) * N
    thr = lam_m * (1 - p[K] / total)
    return dict(rho=min(max(in_serv / N, 0), 1), throughput=thr * 1000, avg_num_in_serv=in_serv, in_sys=in_sys)


def _edge_chains():
    out = []
    wide = wide_fleet()
    for N in (614, 615, 620, 640, 720):
        qa = _analyzer(wide, WIDE_N.index(N), N)
        rmin, rmax = qa.rate_range()
        out.append((f"wide N={N} at RateRange.Max", qa, f32(rmax)))
    qa = _analyzer(raised_fleet(), 0, RAISED_N)
    lam = sweep_lambdas(*qa.rate_range(), RAISED_RATES)[RAISED_IDX[2]]
    out.append(("raised band", qa, f32(lam * f32(1000))))
    fleet = narrow_fleet()
    for s, lam in enumerate(NARROW_LAMBDA[:5]):
        qa = _analyzer(fleet, s, 432)
        out.append((f"narrow batch 432 lambda {lam}", qa, f32(grid_lambda(fleet, s, 1) * f32(1000))))
    return out


@pytest.mark.parametrize("case", range(11))
def test_oracle_matches_200_bit_chain(case):
    """rho, throughput and avgNumInServers of the oracle's Analyze (with the reference's rescale where it applies)
    against the same chain in 200-bit arithmetic without rescale, to 1e-6 relative: the device is compared with the
    oracle only, so this guards against a mistake both could share at extreme scale."""
    name, qa, rate = _edge_chains()[case]
    err, m = qa.analyze(float(rate))
    assert err == 0, name
    lam = f32(rate / f32(1000))
    want = _mp_stats(qa.serv_rate(), qa.max_batch, qa.K, lam)
    for k in ("rho", "throughput", "avg_num_in_serv"):
        w = float(want[k])
        assert abs(m[k] - w) <= 1e-6 * abs(w) + 1e-30, f"{name}: {k} {m[k]!r} vs 200-bit {w!r}"
