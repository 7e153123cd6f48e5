#!/usr/bin/env python
"""bench.py — headline benchmark of the WVA optimizer hot path on B200.

Workload (BASELINE.json configs[1], the configuration the metric is quoted on):
100 models x 4 accelerator types x 256 batch sizes x 64 replica levels = 6,553,600
candidate allocations per step per GPU (synthetic fleet, SURVEY.md §8d, PCG64 seed 42).
One step = one pass of the hot path over that grid: state-dependent M/M/1/K evaluation
of every cell + SLO feasibility + cost + transition penalty + per-model argmin.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras] [--dump-outputs DIR]

N > 1 is launched by torchrun, one rank per GPU: the fleet is sharded by model (weak
scaling: 100 models per GPU), the only exchange is ONE NCCL all-gather of the per-shard
winner records (40 B per model) after the local solve.

The JSON line printed by rank 0 follows the driver's contract; `value` is device-resident
throughput (inputs already in HBM), `e2e` goes through the C ABI with host buffers
(H2D of the fleet + D2H of the winners inside the timed region).  `extras` carries the other
BASELINE configurations (single VA, latency sweep, 10k-server min-cost solve — sharded when
N > 1 —, streaming re-solve), each with its own CPU sample.
"""
from __future__ import annotations

import argparse
import datetime
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "candidate allocations/sec"
UNIT = "candidates/s"
N_MODELS, N_ACC, N_BATCH, N_REPLICAS = 100, 4, 256, 64
ALGO_BYTES_PER_CELL = 100.0   # SURVEY.md §8d: compulsory I/O per candidate (HBM view)
ALGO_F64_PER_STATE = 7.0      # SURVEY.md §8d: reference fp64 ops per state (K mul, 2K div, 4K add/mul)
# Steps run before the timed region so that the 100 ms nvidia-smi samples see this workload.  A FIXED count
# on every rank: the round-1 wall-clock loop let ranks disagree by one all_gather (rank 0 also spawned
# nvidia-smi) and NCCL spun until its watchdog aborted the N = 8 run.
PRE_ROLL_STEPS = 3000


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=("ours", "reference"))
    ap.add_argument("--cpu-sample-pairs", type=int, default=12,
                    help="(model, accelerator) pairs (16384 cells each) per repetition of cpu_baseline (5 repetitions)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary BASELINE configurations")
    ap.add_argument("--ref-seconds", type=float, default=90.0,
                    help="--impl reference: the per-step sample is sized so that the whole run takes about this long")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="--impl ours: after the timed steps, write the winner records of the last timed step as "
                         "DIR/winner_<column>.npy (integer columns as float64, float columns as float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload(rank: int):
    from workload_variant_autoscaler_b200 import config2_grid, synth_fleet
    # weak scaling = fixed work per GPU: every rank draws its 100 models from the same seeded stream (the
    # grid kernel's time varies by +-30 % with the draw, which would otherwise be measured as 'scaling')
    fleet = synth_fleet(N_MODELS, N_ACC, seed=42)
    grid = config2_grid(N_BATCH, N_REPLICAS)
    return fleet, grid


def config_dict(n_gpus: int) -> dict:
    return {
        "workload": "BASELINE configs[1]: 100 models x 4 accelerator types x 256 batch sizes x 64 replica levels "
                    "per GPU, state-dependent M/M/1/K Analyze per cell + per-model min-value SLO-feasible argmin",
        "cells_per_gpu": N_MODELS * N_ACC * N_BATCH * N_REPLICAS,
        "models_per_gpu": N_MODELS, "accelerators": N_ACC, "batch_sizes": N_BATCH, "replica_levels": N_REPLICAS,
        "mean_states_per_cell": 11 * (N_BATCH + 1) / 2,
        "seed": 42, "l2_flush_between_steps": True,
        "parallelism": (f"dp{n_gpus} over models, one all-gather of the winner blocks per step; the gather runs on a side stream and "
                        "overlaps the next step's solve (double-buffered blocks; the timed region ends when the last "
                        "gather has completed)") if n_gpus > 1 else "single GPU",
        "cell_table_materialised": False,
    }


def git_sha() -> str:
    try:
        return subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True,
                              timeout=5).stdout.strip() or "unknown"
    except Exception:
        return "unknown"


def host_info() -> dict:
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return {"cpu_model": model, "logical_cpus": os.cpu_count(), "affinity_cpus": len(os.sched_getaffinity(0))}


# ----------------------------------------------------------------------------
# clocks: sample nvidia-smi during the timed region
# ----------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index),
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 6:
                self.samples.append(parts)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for p in self.samples:
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for n, v in zip(names, p[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------
# CPU legs (the only places bench.py executes oracle/)
# ----------------------------------------------------------------------------
def _cpu_worker(args):
    rank_seed, pairs = args
    import oracle
    from workload_variant_autoscaler_b200 import config2_grid, synth_fleet
    fleet = synth_fleet(N_MODELS, N_ACC, seed=rank_seed)
    grid = config2_grid(N_BATCH, N_REPLICAS)
    per = N_BATCH * N_REPLICAS
    n = 0
    for p in pairs:
        oracle.grid_cells(fleet, grid, p * per, (p + 1) * per)
        n += per
    return n


_REF = {}


def _ref_init():
    import oracle
    from workload_variant_autoscaler_b200 import config2_grid, synth_fleet
    _REF["oracle"] = oracle
    _REF["fleet"] = synth_fleet(N_MODELS, N_ACC, seed=42)
    _REF["grid"] = config2_grid(N_BATCH, N_REPLICAS)


def _ref_task(task):
    p, c0, c1 = task
    per = N_BATCH * N_REPLICAS
    _REF["oracle"].grid_cells(_REF["fleet"], _REF["grid"], p * per + c0, p * per + c1)
    return c1 - c0


def cpu_quota_cores():
    """CPU time the cgroup grants, in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited / unknown."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if q == "max" else float(q) / float(per)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else q / per
    except Exception:
        return None


def sample_pairs(n_pairs: int):
    total = N_MODELS * N_ACC
    n_pairs = max(1, min(n_pairs, total))
    return [int(i * total / n_pairs) for i in range(n_pairs)]


def _pinned_child(conn, cpu, pairs, reps):
    """One process pinned to one core (taskset -c <cpu>): `reps` timed passes over the same sample."""
    try:
        os.sched_setaffinity(0, {cpu})
    except Exception:
        pass
    _cpu_worker((42, pairs[:1]))  # warm caches / page in
    times = []
    n = 0
    for _ in range(reps):
        t0 = time.perf_counter()
        n = _cpu_worker((42, pairs))
        times.append(time.perf_counter() - t0)
    conn.send((n, times))
    conn.close()


def cpu_baseline_port(n_pairs: int, reps: int = 5) -> dict:
    """Oracle (C port of the Go reference) on ONE pinned core: median of `reps` passes over a bounded sample
    of the same workload (SURVEY.md §8d: taskset -c <cpu>, median of >= 5)."""
    import multiprocessing as mp

    import oracle
    oracle.lib()  # loaded before the workers fork; build() compiled it
    pairs = sample_pairs(n_pairs)
    cpu = sorted(os.sched_getaffinity(0))[0]
    ctx = mp.get_context("fork")
    parent, child = ctx.Pipe()
    pr = ctx.Process(target=_pinned_child, args=(child, cpu, pairs, reps))
    pr.start()
    n, times = parent.recv()
    pr.join()
    med = statistics.median(times)
    return {"value": n / med, "unit": UNIT, "cores": 1, "kind": "port", "pinned_cpu": cpu, "reps": reps,
            "rep_seconds": [round(t, 3) for t in times], **host_info(),
            "sample": f"{len(pairs)} of {N_MODELS * N_ACC} (model, accelerator) pairs x all 256x64 cells "
                      f"= {n} cells per pass, median of {reps} passes ({med:.2f} s) on one core pinned with "
                      f"sched_setaffinity; C restatement of the Go reference (single goroutine), "
                      f"not the Go binary (no Go toolchain on the box)"}


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port; Go cannot be built here) on all host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp

    import oracle
    oracle.lib()  # loaded before the workers fork; build() compiled it
    cores = len(os.sched_getaffinity(0))  # every logical CPU the process may use
    quota = cpu_quota_cores()            # ... unless a cgroup quota caps the CPU time below that
    per_pair = N_BATCH * N_REPLICAS
    task_cells = 2048
    # one-core rate on a small sample, so that the record shows what the process pool actually gained
    one = cpu_baseline_port(4, reps=3)
    ctx = mp.get_context("fork")
    # one worker per CPU the process can actually get: 128 workers on a 16-core quota only add context switches
    n_proc = cores if not quota else max(1, min(cores, int(round(quota))))
    with ctx.Pool(n_proc, initializer=_ref_init) as pool:
        def run(pairs):
            # tasks of 2048 cells that the workers pull one at a time (the cost of a cell varies 100x with the pair
            # and the rate: static chunks left most workers waiting for the slowest pair)
            tasks = [(p, c0, min(c0 + task_cells, per_pair)) for p in pairs for c0 in range(0, per_pair, task_cells)]
            t0 = time.perf_counter()
            n = sum(pool.map(_ref_task, tasks, chunksize=1))
            return n, time.perf_counter() - t0
        # a step = a bounded sample of the workload: evenly spaced (model, accelerator) pairs, all 256 x 64 cells of
        # each; the sample is sized from a calibration pass so that the whole run takes about --ref-seconds on this host
        n_cal, t_cal = run(sample_pairs(min(max(cores // 2, 8), N_MODELS * N_ACC)))
        rate = n_cal / t_cal
        budget_s = args.ref_seconds / (args.steps + max(args.warmup, 1))
        n_pairs = int(min(max(rate * budget_s / per_pair, 8), N_MODELS * N_ACC))
        pairs_per_step = sample_pairs(n_pairs)
        per_step_cells = len(pairs_per_step) * per_pair
        for _ in range(max(args.warmup, 1)):
            run(pairs_per_step)
        dt = 0.0
        for _ in range(args.steps):
            dt += run(pairs_per_step)[1]
    value = per_step_cells * args.steps / dt
    sample = (f"each step = {len(pairs_per_step)} of {N_MODELS * N_ACC} (model, accelerator) pairs x all 256x64 cells "
              f"= {per_step_cells} cells in tasks of {task_cells}, pulled by {n_proc} worker processes on {cores} usable "
              f"logical CPUs; "
              f"C restatement of the Go reference "
              f"(the Go path itself is single-goroutine and cannot be built here: no Go toolchain)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_dict(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "processes": n_proc, "cpu_quota_cores": quota, "kind": "port",
                         "sample": sample, **host_info(), "one_core_value": one["value"],
                         "parallel_speedup": value / one["value"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------
# Secondary BASELINE configurations (extras)
# ----------------------------------------------------------------------------
def _median_ms(fn, reps=5, warm=1):
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts)


def extras_single_gpu(eng) -> dict:
    """BASELINE configs[0], [2], [3], [4] on one GPU, each through the public API with host buffers (e2e) and
    with a bounded CPU sample of the same work (oracle port, one core)."""
    import oracle
    from workload_variant_autoscaler_b200 import synth_fleet
    from workload_variant_autoscaler_b200.fleet import CONFIG1_LOADS, config1_fleet
    out = {}

    # configs[0]: the single VariantAutoscaling of the emulator sample (one candidate, N = 4): latency per reconcile
    fleets = [config1_fleet(rpm, 0, 278) for rpm in CONFIG1_LOADS]
    same = True
    for f in fleets:
        _, wg = eng.solve(f)
        _, wo = oracle.solve(f)
        same = same and int(wg.replicas[0]) == int(wo["replicas"][0]) and \
            wg.itl.view(np.uint32)[0] == np.float32(wo["itl"][0]).view(np.uint32)
    gpu_ms = _median_ms(lambda: [eng.solve(f) for f in fleets], reps=7) / len(fleets)
    cpu_ms = _median_ms(lambda: [oracle.solve(f) for f in fleets], reps=7) / len(fleets)
    out["config0_single_va"] = {
        "workload": "BASELINE configs[0]: one VariantAutoscaling (A100, N = 4, Premium SLO), loads 0..1440 req/min",
        "gpu_ms_per_reconcile_e2e": gpu_ms, "cpu_oracle_ms_per_reconcile": cpu_ms, "decisions_equal_oracle": bool(same),
        "note": "one candidate cannot fill a GPU: the device path is launch/latency bound here; the CPU port wins "
                "below a few hundred candidates (reported, not hidden)"}

    # configs[2]: latency sweep, 1000 models x 8 accelerator types x 256 rates
    f = synth_fleet(1000, 8, seed=43, max_batch_choices=(4, 8, 16, 32, 64, 128, 256, 512))
    n = f.n_servers * f.n_acc * 256
    ms = _median_ms(lambda: eng.sweep(f, 256), reps=3)
    k_ms = eng.last_kernel_ms
    sub = f.take_servers(np.arange(0, 1000, 125))  # 8 servers x 8 accelerators x 256 rates on the CPU
    t0 = time.perf_counter()
    oracle.sweep(sub, 256)
    cpu_s = time.perf_counter() - t0
    n_sub = sub.n_servers * sub.n_acc * 256
    out["config2_sweep"] = {
        "workload": "BASELINE configs[2]: 1000 models x 8 accelerator types, Analyze at 256 rates per pair",
        "solves": n, "e2e_ms": ms, "kernel_ms": k_ms, "solves_per_s_e2e": n / (ms * 1e-3),
        "solves_per_s_kernel": n / (k_ms * 1e-3),
        "cpu_baseline": {"value": n_sub / cpu_s, "unit": "solves/s", "cores": 1, "kind": "port",
                         "sample": f"{n_sub} solves (8 of the 1000 servers) in {cpu_s:.2f} s"}}

    # configs[3]: 10,000 servers x 8 accelerators, unlimited min-cost assignment (single GPU)
    f = synth_fleet(10000, 8, seed=44, max_batch_choices=(4, 8, 16, 32, 64, 128, 256, 512))
    n = f.n_servers * f.n_acc
    ms = _median_ms(lambda: eng.solve(f, want_candidates=False), reps=3)
    dev_ms = eng.last_device_ms
    sub = f.take_servers(np.arange(0, 10000, 200))  # 50 servers on the CPU
    t0 = time.perf_counter()
    oracle.solve(sub)
    cpu_s = time.perf_counter() - t0
    out["config3_min_cost_10k"] = {
        "workload": "BASELINE configs[3]: 10,000 servers x 8 accelerators, CreateAllocation per candidate + SolveUnlimited",
        "size_candidates": n, "e2e_ms": ms, "device_ms": dev_ms, "candidates_per_s_e2e": n / (ms * 1e-3),
        "cpu_baseline": {"value": sub.n_servers * sub.n_acc / cpu_s, "unit": "size-candidates/s", "cores": 1,
                         "kind": "port", "sample": f"{sub.n_servers * sub.n_acc} candidates (50 of the 10,000 servers) "
                                                   f"in {cpu_s:.2f} s"}}

    # configs[4]: streaming reconcile, 100k resident candidates, arrival churn per tick
    f = synth_fleet(12500, 8, seed=45, max_batch_choices=(4, 8, 16, 32, 64, 128, 256))
    eng.upload(f)
    rng = np.random.default_rng(5)
    eng.resolve()
    lat = []
    for _ in range(32):
        f.srv_arrival_rpm[:] = (f.srv_arrival_rpm * np.exp(rng.normal(0, 0.1, f.n_servers))).astype(np.float32)
        t0 = time.perf_counter()
        eng.update_load(arrival_rpm=f.srv_arrival_rpm)
        eng.resolve()
        lat.append((time.perf_counter() - t0) * 1e3)
    lat = np.array(lat[2:])
    out["config4_streaming"] = {
        "workload": "BASELINE configs[4]: 100,000 resident size candidates, arrival rates x exp(N(0, 0.1^2)) per tick, "
                    "H2D 50 KB + re-solve + D2H winners per tick",
        "size_candidates": f.n_servers * f.n_acc, "tick_ms_p50": float(np.percentile(lat, 50)),
        "tick_ms_p99": float(np.percentile(lat, 99)), "holds_10hz": bool(np.percentile(lat, 99) < 100.0),
        "ticks": int(lat.size)}
    return out


def extras_sharded(eng, rank, world, dev) -> dict:
    """BASELINE configs[3] across `world` GPUs: servers sharded round-robin (Fleet.shard), every rank solves its
    shard on its GPU, ONE NCCL all-gather of the winner records; the gathered solution must equal the single-GPU
    solve of the whole fleet."""
    import torch
    import torch.distributed as dist

    from workload_variant_autoscaler_b200 import synth_fleet
    from workload_variant_autoscaler_b200.parallel import solve_sharded, torch_all_gather

    f = synth_fleet(10000, 8, seed=44, max_batch_choices=(4, 8, 16, 32, 64, 128, 256, 512))
    ag = torch_all_gather(device=dev)

    def local(shard):
        return eng.solve(shard, want_candidates=False)[1]

    win = solve_sharded(local, f, rank=rank, world=world, all_gather=ag)  # warm-up (tables, NCCL buffers)
    ts = []
    for _ in range(3):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        win = solve_sharded(local, f, rank=rank, world=world, all_gather=ag)
        torch.cuda.synchronize()
        t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ts.append(float(t.item()) * 1e3)
    _, full = eng.solve(f, want_candidates=False)
    t0 = time.perf_counter()
    eng.solve(f, want_candidates=False)
    single_ms = (time.perf_counter() - t0) * 1e3
    equal = all(np.array_equal(getattr(win, n).view(np.uint8), getattr(full, n).view(np.uint8))
                for n in ("feasible", "acc", "replicas", "batch", "cost", "value", "itl", "ttft", "rho", "max_rate"))
    ok = torch.tensor([1 if equal else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    return {"workload": "BASELINE configs[3]: 10,000 servers x 8 accelerators sharded over the ranks (Fleet.shard), "
                        "local solve + one all-gather of winners",
            "n_gpus": world, "sharded_ms": statistics.median(ts), "single_gpu_ms_same_box": single_ms,
            "winners_equal_single_gpu_solve": bool(int(ok.item()) == 1), "size_candidates": f.n_servers * f.n_acc}


# ----------------------------------------------------------------------------
# GPU leg
# ----------------------------------------------------------------------------
def dump_winners(block: np.ndarray, n_servers: int, out_dir: str) -> None:
    """One device winner block (int32 [10 * S]: a slot of S words per column of ALLOC_COLUMNS, the feasible flags in
    the first S bytes of theirs) -> out_dir/winner_<column>.npy, integer columns widened to float64 (exact)."""
    from workload_variant_autoscaler_b200._abi import ALLOC_COLUMNS
    os.makedirs(out_dir, exist_ok=True)
    slots = block.reshape(len(ALLOC_COLUMNS), n_servers)
    for k, (name, dt) in enumerate(ALLOC_COLUMNS):
        col = slots[k].view(np.uint8)[:n_servers] if dt is np.uint8 else slots[k].view(dt)
        np.save(os.path.join(out_dir, f"winner_{name}.npy"), col if dt is np.float32 else col.astype(np.float64))


def run_ours(args):
    import torch
    import torch.distributed as dist

    from workload_variant_autoscaler_b200 import Engine, _abi, synth_fleet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # a mismatched collective fails in 90 s instead of NCCL's 10 min watchdog
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=90))
    eng = Engine(local_rank)
    fleet, grid = workload(rank)
    S = fleet.n_servers
    n_cells = S * fleet.n_acc * grid.batch.size * grid.replicas.size

    # device-resident winner blocks: 10 columns x S x 4 B (the feasible column uses S bytes of its slot); two of
    # them, so that the all-gather of step k (side stream) overlaps the solve of step k + 1
    ext = torch.cuda.ExternalStream(eng.stream, device=dev)
    import ctypes as C

    def winner_block():
        t = torch.zeros(10 * S, dtype=torch.int32, device=dev)
        b = t.data_ptr()
        c = _abi.AllocsC()
        c.feasible = C.cast(b, _abi.u8p)
        for k, name in enumerate(("acc", "replicas", "batch"), start=1):
            setattr(c, name, C.cast(b + 4 * S * k, _abi.i32p))
        for k, name in enumerate(("cost", "value", "itl", "ttft", "rho", "max_rate"), start=4):
            setattr(c, name, C.cast(b + 4 * S * k, _abi.f32p))
        return t, c
    blocks = [winner_block(), winner_block()]
    win_local, cols = blocks[0]
    base = win_local.data_ptr()
    gathered = [torch.zeros(10 * S * world, dtype=torch.int32, device=dev) for _ in range(2)] if world > 1 else None
    win_all = gathered[0] if world > 1 else None
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    eng.upload(fleet)  # inputs resident in HBM before the timed region

    # N > 1: one all-gather of the 4 KB winner blocks per step.  Default: NCCL.  WVA_BENCH_PEER=1 selects the
    # library's own exchange kernel (wva_xchg_publish: NVLink stores into every peer's buffer + epoch flags, one
    # launch); measured at N = 2 it is as fast as NCCL's low-latency path (0.405 vs 0.403 ms/step), so the
    # proven collective stays the default.
    xchg, exchange = None, "none (single GPU)"
    if world > 1:
        exchange = "nccl all_gather_into_tensor"
        try:
            if not os.environ.get("WVA_BENCH_PEER"):
                raise RuntimeError("not requested")
            from workload_variant_autoscaler_b200.parallel import PeerExchange
            xchg = PeerExchange(eng, win_local.numel() * 4)
            exchange = "peer-memory kernel (wva_xchg_publish): NVLink stores + epoch flags, one launch"
        except Exception as exc:  # noqa: BLE001 - report and use the library collective
            xchg = None
            if os.environ.get("WVA_BENCH_PEER"):
                exchange += f" (peer exchange unavailable: {exc})"
        ok = torch.tensor([1 if xchg is not None else 0], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            xchg = None

    def step_device():
        eng.grid_solve_device(grid, cols)
        if world > 1:
            if xchg is not None:
                xchg.publish(base)
            else:
                dist.all_gather_into_tensor(win_all, win_local)

    if xchg is not None:
        # one checked step: the peer exchange must deliver exactly what the library collective delivers
        class _Raw:  # zero-copy view of the gathered device buffer
            def __init__(self, ptr, n):
                self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 3}
        with torch.cuda.stream(ext):
            eng.grid_solve_device(grid, cols)
            gptr, stride = xchg.publish(base)
            dist.all_gather_into_tensor(win_all, win_local)
        torch.cuda.synchronize()
        got = torch.as_tensor(_Raw(gptr, world * stride // 4), device=dev).view(world, stride // 4)[:, : win_local.numel()]
        if xchg.error() or not torch.equal(got.reshape(-1), win_all):
            raise SystemExit("peer exchange delivered a different gathered block than NCCL")

    def timed_steps(k):
        """K steps, each timed with CUDA events on the launching stream; L2 flushed in between."""
        evs = []
        with torch.cuda.stream(ext):
            for _ in range(k):
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                step_device()
                e1.record()
                evs.append((e0, e1))
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    step_no = [0]

    def overlapped_steps(k):
        """N > 1, NCCL path: the all-gather of step i runs on a side stream DURING the solve of step i + 1
        (double-buffered winner / gathered blocks).  Timing stays per step with CUDA events on the engine's stream:
        the gather of step i is released only after the L2 flush that precedes step i + 1 (so it cannot hide in the
        untimed flush) and step i + 1's closing event waits for it, i.e. every gather lies inside a timed interval;
        the last step's gather is a timed tail added to the last step."""
        evs = []
        prev = None
        with torch.cuda.stream(ext):
            def release_gather(b):
                go = torch.cuda.Event()
                go.record(ext)
                comm_stream.wait_event(go)
                with torch.cuda.stream(comm_stream):
                    dist.all_gather_into_tensor(gathered[b], blocks[b][0])
                    gone = torch.cuda.Event()
                    gone.record(comm_stream)
                return gone
            for _ in range(k):
                b = step_no[0] & 1
                step_no[0] += 1
                flush.fill_(1)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                gone = release_gather(prev) if prev is not None else None
                eng.grid_solve_device(grid, blocks[b][1])
                if gone is not None:
                    ext.wait_event(gone)
                e1.record()
                evs.append((e0, e1))
                prev = b
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            ext.wait_event(release_gather(prev))
            t1.record()
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in evs]
        ms[-1] += t0.elapsed_time(t1)
        return ms
    overlap = world > 1 and xchg is None and not os.environ.get("WVA_BENCH_NO_OVERLAP")
    run_steps = overlapped_steps if overlap else timed_steps

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # off the ranks' common path: nothing below depends on when it comes up
    timed_steps(max(args.warmup, 3))

    # multi-GPU self-check: every rank holds the same fleet, so every slot of the gathered block must equal this
    # rank's own winner block, bit for bit (a broken exchange cannot hide behind a plausible number)
    gather_check = None
    if world > 1 and xchg is None:
        same = torch.equal(win_all.view(world, -1), win_local.view(1, -1).expand(world, -1))
        okc = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(okc, op=dist.ReduceOp.MIN)
        gather_check = bool(int(okc.item()) == 1)
        if not gather_check:
            raise SystemExit("all-gathered winner blocks differ from the locally computed block")

    # a step is < 1 ms: keep the same load running before the timed region so that the 100 ms nvidia-smi samples
    # are taken under this workload (they continue through the timed region); fixed step count on every rank
    def block_ms():
        t = torch.tensor([sum(run_steps(100))], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # the same number on every rank: identical decisions below
        return float(t.item())
    prev = None
    for _ in range(PRE_ROLL_STEPS // 100):
        prev = block_ms()
    # ... and until the box has settled: two consecutive 100-step blocks within 2 % (a run started right after another
    # job on the same GPUs was once 6 % slow for its whole timed region); bounded, and decided on the all-reduced
    # time, so every rank runs the same number of blocks
    settle_blocks = 0
    for _ in range(60):
        cur = block_ms()
        settle_blocks += 1
        if abs(cur - prev) <= 0.02 * prev:
            break
        prev = cur
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = eng.launch_count
    wall0 = time.perf_counter()
    per_step = run_steps(args.steps)
    torch.cuda.synchronize()
    if overlap:  # the overlapped gathers delivered the same blocks (both buffers were used)
        same = all(torch.equal(gathered[b].view(world, -1), blocks[b][0].view(1, -1).expand(world, -1)) for b in (0, 1))
        okc = torch.tensor([1 if same else 0], device=dev)
        dist.all_reduce(okc, op=dist.ReduceOp.MIN)
        if int(okc.item()) != 1:
            raise SystemExit("overlapped all-gather delivered blocks that differ from the locally computed ones")
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - wall0
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:  # the block the last timed step wrote (overlapped steps alternate two)
        dump_winners(blocks[(step_no[0] - 1) & 1 if overlap else 0][0].cpu().numpy(), S, args.dump_outputs)
    total_ms = torch.tensor([sum(per_step)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    clocks = sampler.stop() if rank == 0 else None

    # dominant kernel: per-launch device time measured live (CUDA events on the engine's stream)
    def kernel_ms_of(fl, reps=5):
        ks = []
        for _ in range(reps):
            with torch.cuda.stream(ext):
                flush.fill_(1)
            torch.cuda.synchronize()
            eng.grid_solve(fl, grid)  # records the grid kernel's own event pair
            ks.append(eng.last_kernel_ms)
        return statistics.median(ks)
    kernel_ms = kernel_ms_of(fleet)

    # e2e through the C ABI with host buffers (H2D fleet + D2H winners inside the timed region)
    from workload_variant_autoscaler_b200._abi import Allocs
    win = Allocs(fleet.n_servers)  # a reconcile loop keeps one winner block and hands it to every call
    for _ in range(2):
        eng.grid_solve(fleet, grid, out=win)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.grid_solve(fleet, grid, out=win)
    e2e_s = time.perf_counter() - t0
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_t.item())
    h2d = sum(getattr(fleet, n).nbytes for n in fleet._F32 + fleet._I32 + fleet._U8) + grid.batch.nbytes * 2 + \
        grid.replicas.nbytes
    d2h = sum(v.nbytes for v in win.columns().values()) + 32

    # seed sensitivity of the dominant kernel (the headline is quoted on seed 42, SURVEY.md §8d)
    seed_ms = None
    if world == 1 and not args.no_extras:
        seed_ms = {}
        for seed in range(42, 50):
            seed_ms[str(seed)] = kernel_ms_of(synth_fleet(N_MODELS, N_ACC, seed=seed), reps=3)
        eng.upload(fleet)

    extras = None
    if not args.no_extras:
        if world == 1:
            smp = ClockSampler(local_rank)
            smp.start()
            extras = extras_single_gpu(eng)
            extras["clocks"] = smp.stop()
        else:
            extras = {"config3_min_cost_10k_sharded": extras_sharded(eng, rank, world, dev)}

    if rank == 0:
        peaks, prof = {}, {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        try:  # ncu-derived figures of the dominant kernel (profiles/, committed per round)
            prof = json.load(open(os.path.join(ROOT, "profiles", "roofline_latest.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        achieved = ALGO_BYTES_PER_CELL * n_cells / (kernel_ms * 1e-3) / 1e9
        ms_per_step = total_ms / args.steps
        achieved_step = ALGO_BYTES_PER_CELL * n_cells / (ms_per_step * 1e-3) / 1e9
        states = float(config_dict(1)["mean_states_per_cell"]) * n_cells
        value = n_cells * world * args.steps / (total_ms * 1e-3)
        fp64_peak = float(prof.get("fp64_peak_tdfma_s", 17.07))
        ncu_from = {"capture": prof.get("source"), "capture_git_sha": prof.get("git_sha"), "run_git_sha": git_sha(),
                    "note": "ncu figures are read from the committed capture named here (profiles/), not measured in "
                            "this run; they describe this code only if the two SHAs name the same kernels"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(world),
            "exchange": exchange, "gather_check_equal_local": gather_check,
            "exchange_overlapped_with_next_step": bool(overlap),
            "pre_roll_steps": PRE_ROLL_STEPS + 100 * settle_blocks,
            "e2e": {"value": n_cells * world * args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h),
                    "note": "wva_grid_solve through the C ABI with host buffers: H2D of the fleet (staged through the "
                            "library's pinned arena) and D2H of the winner block inside the timed region"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {
                # the contract's keys, HBM view (SURVEY.md 8d accounting).  The kernel's real limiter is FP64 issue:
                # see bound_actual / fp64 below.
                "bound": "hbm", "bound_actual": "fp64-issue",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "frac_step_level": achieved_step / hbm_peak,
                "traffic": prof.get("grid_kernel_dram_bytes"), "peak_source": peak_src, "kernel": "grid_kernel",
                "kernel_ms": kernel_ms, "ms_per_step": ms_per_step,
                "algorithmic_bytes_per_launch": ALGO_BYTES_PER_CELL * n_cells,
                "note": "achieved = 100 B/cell (SURVEY.md 8d) x cells / live CUDA-event time of grid_kernel alone "
                        "(frac) or of the whole step (frac_step_level).  The 100 B/cell is a notional accounting: "
                        "inputs are factored tables, the kernel's DRAM traffic (traffic, from ncu) is ~1 % of it; "
                        "the binding resource is FP64 issue (fp64.pipe_active_pct_ncu)",
                "ncu_fields_from": ncu_from,
                "fp64": {
                    "peak_tdfma_per_s": fp64_peak, "peak_source": "tools/fp64_peak.cu on this pool (profiles/r01_fp64_peak.txt)",
                    "pipe_active_pct_ncu": prof.get("grid_kernel_fp64_pipe_pct"),
                    "issue_active_pct_ncu": prof.get("grid_kernel_issue_pct"),
                    "reference_ops_per_launch": ALGO_F64_PER_STATE * states,
                    "reference_equivalent_tflops": ALGO_F64_PER_STATE * states / (kernel_ms * 1e-3) / 1e12,
                    "note": "reference_equivalent counts the reference's 7*K float64 ops per solve; it exceeds the "
                            "pipe peak because exact early termination executes ~2% of the reference's state steps "
                            "(DESIGN.md 3.2); pipe_active_pct is what the hardware actually issued",
                },
            },
            "wall_s_timed_region": wall,
        }
        if seed_ms:
            v = sorted(seed_ms.values())
            line["seed_sensitivity"] = {"kernel_ms_by_seed": seed_ms, "min": v[0], "median": statistics.median(v),
                                        "max": v[-1], "note": "grid_kernel ms for the same configuration drawn with "
                                                              "seeds 42..49; the headline uses seed 42 (SURVEY.md 8d)"}
        if extras:
            line["extras"] = extras
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_port(args.cpu_sample_pairs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    eng.close()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
