"""wva_resolve_scenarios against L sequential ticks on the configs[4] streaming fleet (tools/bench_configs.py 5).

For L in {1, 4, 16, 64}: the median host wall time of one resolve_scenarios call (it ends in a synchronise), its
last_kernel_ms / last_device_ms, and the median summed wall time of L update_load + resolve ticks over the same rows,
the two alternated in one process.  --profile adds the per-kernel device time of one L = 16 call and of the 16 ticks
(torch.profiler).  Prints one JSON object; --out also writes it to a file.  Run on the GPU box:

    python tools/scenario_bench.py --out profiles/scenario_bench_<tag>.json
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
from workload_variant_autoscaler_b200 import Engine, synth_fleet  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:  # read-only query
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


def rows_for(base, L, rng):
    """Forecast-like scenarios: every server's rate scaled by its own log-normal factor (sigma 0.3)."""
    return (base[None, :] * np.exp(rng.normal(0.0, 0.3, (L, base.size)))).astype(np.float32)


def ticks(e, rows):
    t0 = time.perf_counter()
    for r in rows:
        e.update_load(arrival_rpm=r)
        e.resolve()
    return time.perf_counter() - t0


def scen(e, rows):
    t0 = time.perf_counter()
    e.resolve_scenarios(rows)
    return time.perf_counter() - t0


def kernel_split(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA":
            k = ev.name.split("(")[0].replace("void ", "").replace("wva::", "")
            d = out.setdefault(k, [0, 0.0])
            d[0] += 1
            d[1] += ev.device_time / 1e3 if hasattr(ev, "device_time") else ev.cuda_time / 1e3
    return {k: {"launches": n, "ms": round(ms, 4)} for k, (n, ms) in sorted(out.items(), key=lambda kv: -kv[1][1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--ls", default="1,4,16,64")
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    name, limit = card()
    e = Engine(0)
    f = synth_fleet(12500, 8, seed=45, max_batch_choices=(4, 8, 16, 32, 64, 128, 256))
    base = f.srv_arrival_rpm.copy()
    e.upload(f)
    e.resolve()
    rng = np.random.default_rng(7)
    res = {"card": name, "power_limit": limit, "fleet": "synth_fleet(12500, 8, seed=45, max_batch 4..256)",
           "pairs": f.n_servers * f.n_acc, "reps": a.reps, "L": {}}
    for L in [int(x) for x in a.ls.split(",")]:
        rows = rows_for(base, L, rng)
        scen(e, rows)  # warm: buffers, tables
        ticks(e, rows)
        ts, tt, kms, dms = [], [], [], []
        for _ in range(a.reps):
            ts.append(scen(e, rows))
            kms.append(e.last_kernel_ms)
            dms.append(e.last_device_ms)
            tt.append(ticks(e, rows))
        r = {"scenarios_ms": 1e3 * float(np.median(ts)), "scenarios_ms_min": 1e3 * float(np.min(ts)),
             "kernel_ms": float(np.median(kms)), "device_ms": float(np.median(dms)),
             "ticks_ms": 1e3 * float(np.median(tt)), "ticks_ms_min": 1e3 * float(np.min(tt))}
        r["ratio"] = r["scenarios_ms"] / r["ticks_ms"]
        res["L"][str(L)] = r
        print(json.dumps({"L": L, **r}), file=sys.stderr)
    if a.profile:
        rows = rows_for(base, 16, rng)
        res["profile_L16"] = {"scenarios": kernel_split(lambda: e.resolve_scenarios(rows)),
                              "ticks": kernel_split(lambda: ticks(e, rows))}
    e.update_load(arrival_rpm=base)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
