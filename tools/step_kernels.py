"""Per-launch device times of the grid pipeline on the flagship workload (BASELINE configs[1], fleet seed 42), from
torch.profiler with CUDA activities, with row resolution on and off (WVA_GRID_ROWRES) in the same process; and how
many rows and cells row resolution covers on that fleet.

    python tools/step_kernels.py [--steps 300] [--out FILE.json]

Steps are issued like bench.py's (device-resident winners, L2 flushed before every step).  A library without the
switch (or without the row diagnostics) runs the same code in both arms and reports no row counts.
"""
import argparse
import collections
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from workload_variant_autoscaler_b200 import Engine, _abi, config2_grid, synth_fleet  # noqa: E402

INT_MAX = 2**31 - 1


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def winner_block(S, dev):
    t = torch.zeros(10 * S, dtype=torch.int32, device=dev)
    b = t.data_ptr()
    c = _abi.AllocsC()
    c.feasible = C.cast(b, _abi.u8p)
    for k, name in enumerate(("acc", "replicas", "batch"), start=1):
        setattr(c, name, C.cast(b + 4 * S * k, _abi.i32p))
    for k, name in enumerate(("cost", "value", "itl", "ttft", "rho", "max_rate"), start=4):
        setattr(c, name, C.cast(b + 4 * S * k, _abi.f32p))
    return t, c


def kernel_medians(eng, grid, cols, steps, dev):
    ext = torch.cuda.ExternalStream(eng.stream, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    with torch.cuda.stream(ext):
        for _ in range(50):
            eng.grid_solve_device(grid, cols)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with torch.cuda.stream(ext):
            for _ in range(steps):
                flush.fill_(1)
                eng.grid_solve_device(grid, cols)
        torch.cuda.synchronize()
    per = collections.defaultdict(list)
    for ev in prof.events():
        m = re.search(r"wva::(\w+)\(", ev.name)
        if m:
            per[m.group(1)].append(ev.time_range.end - ev.time_range.start)
    return {k: {"median_us": statistics.median(v), "launches": len(v)} for k, v in sorted(per.items())}


def row_counts(eng, fleet, grid):
    L = eng._L
    if not hasattr(L, "wva_dbg_read_rows"):
        return None
    L.wva_dbg_read_rows.restype = C.c_longlong
    L.wva_dbg_read_rows.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong]
    eng.grid_solve(fleet, grid)
    S, A, B, R = fleet.n_servers, fleet.n_acc, grid.batch.size, grid.replicas.size
    row_j = np.zeros(S * A * R, np.int32)
    res = np.zeros(S * A * R, np.uint8)
    n = L.wva_dbg_read_rows(eng._h, row_j.ctypes.data, res.ctypes.data, row_j.size)
    assert n == row_j.size
    b = grid.batch.astype(np.int64)
    K = b + b * int(fleet.max_queue_to_batch_ratio)
    jl = row_j.astype(np.int64)
    shared = (jl[:, None] != INT_MAX) & (b[None, :] >= jl[:, None] + 2) & (K[None, :] < (1 << 23))  # [rows, B]
    per_row = shared.sum(axis=1)
    return {"rows": int(row_j.size), "rows_sharing": int((row_j != INT_MAX).sum()), "rows_resolved": int(res.sum()),
            "cells": int(S * A * B * R), "cells_shared": int(per_row.sum()),
            "cells_skipped": int(per_row[res.astype(bool)].sum()),
            "note": "cells_shared: cells whose batch size is past their row's shared chain (analysable or not); "
                    "cells_skipped: those of resolved rows, which grid_sort_local no longer evaluates"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    eng = Engine(0)
    fleet, grid = synth_fleet(100, 4, seed=42), config2_grid()
    eng.upload(fleet)
    _, cols = winner_block(fleet.n_servers, dev)
    out = {"card": card(), "steps": args.steps, "arms": {}}
    for arm in ("1", "0"):
        os.environ["WVA_GRID_ROWRES"] = arm
        out["arms"]["WVA_GRID_ROWRES=" + arm] = kernel_medians(eng, grid, cols, args.steps, dev)
    os.environ["WVA_GRID_ROWRES"] = "1"
    out["rows"] = row_counts(eng, fleet, grid)
    eng.close()
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
