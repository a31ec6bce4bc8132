"""Host-side logic of the range-sharded MSM on CPU: world_size-2 gloo processes partition the
points like Client.hpp:747-787, all-gather their per-rank partial results and rank 0 combines.
The per-rank MSM itself is done with the oracle here (no GPU in this container); what is under
test is the partition, the exchange and the combination."""
import os
import socket
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shard_ranges_cover_everything():
    from porla_b200.sharding import shard_range
    for n in (0, 1, 7, 128, 766, 1 << 20):
        for world in (1, 2, 3, 8):
            seen = []
            for r in range(world):
                lo, hi = shard_range(n, world, r)
                assert 0 <= lo <= hi <= n
                seen.extend(range(lo, hi)) if n <= 1000 else None
                if r:
                    assert lo == prev_hi
                prev_hi = hi
            assert prev_hi == n
            if n <= 1000:
                assert seen == list(range(n))
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


def _worker(rank, world, port, n, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import curves_py as O
    from porla_b200.sharding import gather_window_sums, shard_range
    from tests.common import be, bn254_points, det_scalar
    pts = bn254_points(n)
    sc = [det_scalar(b"porla-sc", i) for i in range(n)]
    lo, hi = shard_range(n, world, rank)
    part = O.msm(O.BN254, sc[lo:hi], pts[lo:hi])
    local = torch.frombuffer(bytearray(O.bn254_marshal(part)), dtype=torch.uint8)
    allp = gather_window_sums(local, world, dist)
    assert allp.numel() == 64 * world
    if rank == 0:
        acc = None
        for r in range(world):
            b = bytes(allp[64 * r:64 * r + 64].numpy().tobytes())
            acc = O.add(O.BN254, acc, O.bn254_unmarshal(b))
        q.put(O.bn254_marshal(acc).hex())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gloo_sharded_msm_matches_single():
    from oracle import curves_py as O
    from tests.common import bn254_points, det_scalar
    n, world = 61, 2
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = O.msm(O.BN254, [det_scalar(b"porla-sc", i) for i in range(n)], bn254_points(n))
    assert got == O.bn254_marshal(want).hex()


def test_sharded_engine_plan_codes():
    """ShardedMsm's plan: one window layout for all ranks (planned for the largest shard); the fixed-base form exchanges
    ONE partial sum per rank under a code that carries the expansion's window size."""
    import porla_b200 as pb
    from porla_b200.sharding import ShardedMsm
    dev = torch.device("cpu")
    e = ShardedMsm(pb.CURVE_BN254, (1 << 20) + 5, 2, 0, dist, dev)
    e1 = ShardedMsm(pb.CURVE_BN254, (1 << 20) + 5, 2, 1, dist, dev)
    assert (e.plan_code, e.nwin) == (e1.plan_code, e1.nwin) and e.nwin > 1
    f = ShardedMsm(pb.CURVE_BN254, 1 << 20, 8, 3, dist, dev, fixed_base_bits=20)
    assert f.nwin == 1 and f.plan_code & 0xff == 20 and f.plan_code & pb.lib.PLAN_FIXED and f.wsum.numel() == 128
