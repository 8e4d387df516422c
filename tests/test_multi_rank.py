"""The N > 1 host logic of bench.py on CPU: two processes over gloo (the data path has no collective: instances are
sharded by index; only the timings and unit counts are reduced)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import bench
    from jrl_walkgen_b200 import workloads
    # every rank builds its own shard of the same global problem set
    lo, hi = workloads.shard_instances(1000, rank, world)
    offsets, z = workloads.preview_batch(4, seed=1000 * rank)
    ms = 10.0 + 5.0 * rank                      # rank 1 is slower
    units = float(hi - lo)
    max_ms, total = bench.reduce_over_ranks(dist, [ms], [units], device="cpu")
    q.put((rank, lo, hi, float(z.sum()), max_ms[0], total[0]))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_shard_and_reduce_over_gloo():
    # torch is imported by the spawned ranks only: in a test process where the library has already dlopen'ed the system's
    # libnccl.so.2 (test_multi_gpu), importing torch here would bind libtorch_cuda to that older NCCL and fail
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, lo0, hi0, s0, m0, t0), (r1, lo1, hi1, s1, m1, t1) = res
    assert (lo0, hi0, lo1, hi1) == (0, 500, 500, 1000)          # disjoint, exhaustive
    assert s0 != s1                                             # per-rank seeds: different walks
    assert m0 == m1 == 15.0 and t0 == t1 == 1000.0              # MAX over ranks of the time, SUM of the units


def test_shard_instances_covers_every_instance_once():
    from jrl_walkgen_b200 import workloads
    for B in (0, 1, 7, 16384, 1000003):
        for world in (1, 2, 4, 8):
            seen = 0
            prev = 0
            for r in range(world):
                lo, hi = workloads.shard_instances(B, r, world)
                assert lo == prev and hi >= lo
                prev = hi; seen += hi - lo
            assert seen == B and prev == B
