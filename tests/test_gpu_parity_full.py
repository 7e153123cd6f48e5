"""GPU parity at BASELINE sizes: the CUDA path (through the C ABI) against the CPU oracle, bit for bit, with the
oracle spread over the box's host cores by a process pool (it is single-threaded, like the reference).

 * configs[1]: ALL 100 models x 4 accelerators x 256 batch sizes x 64 replica levels (6.55 M cells), cells and winners
 * configs[2]: latency sweep with N in {256, 512}, 256 rates, 64 pairs
 * configs[3]: size path on 512 servers x 8 accelerators with N up to 512
 * configs[4]: streaming, 32 ticks with arrival churn and token-statistics changes
 * multi-GPU (needs >= 2 GPUs on the box): the peer-memory exchange kernel against NCCL; the sharded solves
   (unlimited and limited mode) under NCCL against the oracle on the whole fleet
"""
import multiprocessing as mp
import os
import socket
import sys

import numpy as np
import pytest

from tests.util import assert_allocs_equal, assert_f32_bits_equal
from workload_variant_autoscaler_b200 import synth_fleet

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _n_workers():
    return max(1, min(len(os.sched_getaffinity(0)), 64))


# ---- pool workers (fork: the parent's fleet objects are inherited through module globals) ----------------------------
_JOB = {}


def _grid_worker(idx):
    import oracle
    sub = _JOB["fleet"].take_servers(np.asarray(idx))
    cells, win = oracle.grid_solve(sub, _JOB["grid"], want_cells=True)
    return idx, cells, win


def _solve_worker(idx):
    import oracle
    sub = _JOB["fleet"].take_servers(np.asarray(idx))
    cand, win = oracle.solve(sub)
    return idx, cand, win


def _sweep_worker(idx):
    import oracle
    sub = _JOB["fleet"].take_servers(np.asarray(idx))
    return idx, oracle.sweep(sub, _JOB["n_rates"])


def _pool_map(fn, chunks):
    import oracle
    oracle.build()
    ctx = mp.get_context("fork")
    with ctx.Pool(min(_n_workers(), len(chunks))) as pool:
        return pool.map(fn, chunks)


def test_config2_all_models_bit_exact(engine):
    """BASELINE configs[1] in full: every one of the 6,553,600 cells and all 100 winners against the oracle."""
    from workload_variant_autoscaler_b200 import config2_grid
    fleet = synth_fleet(100, 4, seed=42)
    grid = config2_grid()
    _JOB.update(fleet=fleet, grid=grid)
    chunks = [[s] for s in range(fleet.n_servers)]           # one server (65,536 cells, ~1 s) per task
    results = _pool_map(_grid_worker, chunks)
    cells_g, win_g = engine.grid_solve(fleet, grid, want_cells=True)
    _, win_nocells = engine.grid_solve(fleet, grid)          # the bench's path: no cell table, winners recomputed
    per = fleet.n_acc * 256 * 64
    n_ok = 0
    for idx, cells_o, win_o in results:
        s = idx[0]
        sl = slice(s * per, (s + 1) * per)
        assert np.array_equal(cells_g["flags"][sl], cells_o["flags"]), f"server {s}: flags"
        for k in ("ttft", "itl", "rho", "throughput"):
            assert_f32_bits_equal(cells_g[k][sl], cells_o[k], f"server {s}: cells.{k}")
        n_ok += int((cells_o["flags"] & 1).sum())
        for name in ("feasible", "acc", "replicas", "batch"):
            for w in (win_g, win_nocells):
                assert int(np.asarray(getattr(w, name))[s]) == int(win_o[name][0]), (s, name)
        for name in ("cost", "value", "itl", "ttft", "rho", "max_rate"):
            for w in (win_g, win_nocells):
                assert_f32_bits_equal(getattr(w, name)[s:s + 1], win_o[name], f"server {s}: winner {name}")
    assert n_ok > 5_000_000, "most cells of the configuration are analysable"


def test_sweep_large_batches_bit_exact(engine):
    """BASELINE configs[2] shape at parity-checkable size: 16 servers x 4 accelerators = 64 pairs, N in {256, 512},
    256 rates each (16,384 solves of up to 5,632 states)."""
    fleet = synth_fleet(16, 4, seed=61, max_batch_choices=(256, 512))
    n_rates = 256
    _JOB.update(fleet=fleet, n_rates=n_rates)
    results = _pool_map(_sweep_worker, [[s] for s in range(fleet.n_servers)])
    g = engine.sweep(fleet, n_rates)
    per = fleet.n_acc * n_rates
    for idx, o in results:
        s = idx[0]
        sl = slice(s * per, (s + 1) * per)
        assert np.array_equal(g["valid"][sl], o["valid"]), f"server {s}: valid"
        for k in ("rate", "ttft", "itl", "throughput", "rho"):
            assert_f32_bits_equal(g[k][sl], o[k], f"server {s}: sweep.{k}")
    assert g["valid"].mean() > 0.9


def test_size_path_512_servers_bit_exact(engine):
    """BASELINE configs[3] shape: 512 servers x 8 accelerators (4,096 CreateAllocation candidates), batch sizes up to
    512 (K = 5,632), unlimited argmin; candidates and winners against the oracle."""
    fleet = synth_fleet(512, 8, seed=67, max_batch_choices=(4, 8, 16, 32, 64, 128, 256, 512), zero_load_frac=0.05)
    fleet.srv_min_replicas[::9] = 0
    _JOB.update(fleet=fleet)
    chunks = [list(range(s, min(s + 8, fleet.n_servers))) for s in range(0, fleet.n_servers, 8)]
    results = _pool_map(_solve_worker, chunks)
    cand_g, win_g = engine.solve(fleet)
    A = fleet.n_acc
    from workload_variant_autoscaler_b200._abi import ALLOC_COLUMNS, Allocs
    for idx, cand_o, win_o in results:
        s0, n = idx[0], len(idx)
        sub_c, sub_w = Allocs(n * A), Allocs(n)
        for name, _ in ALLOC_COLUMNS:
            getattr(sub_c, name)[:] = getattr(cand_g, name)[s0 * A:(s0 + n) * A]
            getattr(sub_w, name)[:] = getattr(win_g, name)[s0:s0 + n]
        assert_allocs_equal(sub_c, cand_o, f"servers {s0}..: size candidates")
        assert_allocs_equal(sub_w, win_o, f"servers {s0}..: winners")
    assert cand_g.feasible.sum() > 2000 and (cand_g.batch >= 256).sum() > 200


def test_streaming_32_ticks_with_token_changes(engine, oracle_mod):
    """BASELINE configs[4] shape: a resident fleet re-solved tick after tick; arrival rates drift every tick, the
    token statistics of some servers change every fourth tick (tables rebuilt), some servers fall to zero load and
    come back.  Every tick's winners equal a fresh oracle solve of the same fleet."""
    fleet = synth_fleet(48, 4, seed=71, keep_accelerator=True, max_batch_choices=(4, 8, 16, 32, 64))
    engine.upload(fleet)
    rng = np.random.default_rng(7)
    base = fleet.srv_arrival_rpm.copy()
    for tick in range(32):
        fleet.srv_arrival_rpm[:] = (fleet.srv_arrival_rpm * np.exp(rng.normal(0, 0.1, fleet.n_servers))).astype(np.float32)
        if tick % 5 == 2:
            fleet.srv_arrival_rpm[tick % fleet.n_servers] = 0.0          # a server goes idle ...
        if tick % 5 == 4:
            z = fleet.srv_arrival_rpm == 0
            fleet.srv_arrival_rpm[z] = base[z]                           # ... and comes back
        kw = {"arrival_rpm": fleet.srv_arrival_rpm}
        if tick % 4 == 3:
            pick = rng.integers(0, fleet.n_servers, 6)
            fleet.srv_in_tokens[pick] = rng.integers(16, 2049, 6)
            fleet.srv_out_tokens[pick] = rng.integers(16, 1025, 6)
            kw.update(in_tokens=fleet.srv_in_tokens, out_tokens=fleet.srv_out_tokens)
        engine.update_load(**kw)
        _, win_g = engine.resolve()
        _, win_o = oracle_mod.solve(fleet)
        assert_allocs_equal(win_g, win_o, f"tick {tick}")


# ---- multi-GPU: the peer exchange kernel against NCCL ---------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _peer_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import datetime

    import torch
    import torch.distributed as dist

    from workload_variant_autoscaler_b200 import Engine
    from workload_variant_autoscaler_b200.parallel import PeerExchange
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
    eng = Engine(rank)
    n = 1000  # int32 words per rank's block
    x = PeerExchange(eng, 4 * n)
    ext = torch.cuda.ExternalStream(eng.stream, device=dev)
    ok = True
    for step in range(5):
        block = (torch.arange(n, dtype=torch.int32, device=dev) * (rank + 1) + 1000 * step)
        torch.cuda.synchronize()
        with torch.cuda.stream(ext):
            gptr, stride = x.publish(block.data_ptr())
        eng.synchronize()
        want = torch.empty(world * n, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(want, block)

        class _Raw:
            def __init__(self, ptr, cnt):
                self.__cuda_array_interface__ = {"shape": (cnt,), "typestr": "<i4", "data": (ptr, False), "version": 3}
        got = torch.as_tensor(_Raw(gptr, world * stride // 4), device=dev).view(world, stride // 4)[:, :n].reshape(-1)
        ok = ok and bool(torch.equal(got, want)) and x.error() == 0
    open(os.path.join(out_dir, f"rank{rank}.txt"), "w").write("ok" if ok else "mismatch")
    dist.barrier()
    x.close()
    eng.close()
    dist.destroy_process_group()


def test_peer_exchange_matches_nccl(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    import torch.multiprocessing as tmp_mp
    world = 2
    tmp_mp.spawn(_peer_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(os.path.join(tmp_path, f"rank{r}.txt")).read() == "ok"


# ---- multi-GPU: the product's sharded solves (unlimited and limited mode) against the oracle on the whole fleet --------
def _sharded_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import datetime

    import torch
    import torch.distributed as dist

    import oracle
    from workload_variant_autoscaler_b200 import Engine
    from workload_variant_autoscaler_b200._abi import SAT_PRIORITY_ROUND_ROBIN
    from workload_variant_autoscaler_b200.parallel import solve_sharded, solve_sharded_limited, torch_all_gather
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev, timeout=datetime.timedelta(seconds=120))
    eng = Engine(rank)
    ag = torch_all_gather(device=dev)
    msg = "ok"
    try:
        # unlimited mode: shards solve independently, one all-gather of the winner records
        f = synth_fleet(203, 4, seed=31, max_batch_choices=(4, 8, 16, 32, 64), zero_load_frac=0.1)
        win = solve_sharded(lambda sh: eng.solve(sh)[1], f, rank=rank, world=world, all_gather=ag)
        _, win_o = oracle.solve(f)
        assert_allocs_equal(win, win_o, f"rank {rank}: sharded unlimited winners")
        # limited mode: shards size their candidates, one all-gather of the tables, the same greedy pass on every rank
        g = synth_fleet(61, 3, seed=32, max_batch_choices=(2, 4, 8, 16), zero_load_frac=0.1)
        g.unlimited = False
        g.saturation_policy = SAT_PRIORITY_ROUND_ROBIN
        g.delayed_best_effort = True
        g.type_capacity[:] = 30
        g.srv_priority[:] = np.random.default_rng(3).choice([1, 5, 10], g.n_servers)
        cand, win = solve_sharded_limited(lambda sh: eng.analyze(sh), g, rank=rank, world=world, all_gather=ag)
        cand_o, win_o = oracle.solve(g)
        assert_allocs_equal(win, win_o, f"rank {rank}: sharded limited winners")
        assert_allocs_equal(cand, cand_o, f"rank {rank}: sharded limited candidates")
    except AssertionError as exc:
        msg = str(exc)[:500]
    open(os.path.join(out_dir, f"rank{rank}.txt"), "w").write(msg)
    dist.barrier()
    eng.close()
    dist.destroy_process_group()


def test_sharded_solves_on_two_gpus_match_the_oracle(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    import torch.multiprocessing as tmp_mp
    world = 2
    tmp_mp.spawn(_sharded_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(os.path.join(tmp_path, f"rank{r}.txt")).read() == "ok"
