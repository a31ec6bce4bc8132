"""The in-call multi-GPU partition (multi.cu; the reference's 8-thread range partition of Client.hpp:747-787 with devices in
place of threads), the pageable-buffer copy pool, and the one-process-per-GPU sharded path over NCCL.

Tests that need two real devices skip on a one-GPU box; the partition logic itself is exercised everywhere by letting
several parts share device 0 (PORLA_OVERSUBSCRIBE_DEVICES=1: each part still has its own worker thread, stream, staging
buffers and window sums)."""
import ctypes as C
import hashlib
import os
import random
import socket
import sys

import pytest

import porla_b200 as pb
from oracle import curves_py as O
from oracle import loader

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BN = O.BN254


def _inputs(n, seed, with_infinity=True):
    G = O.bn254_marshal((1, 2))
    step = O.bn254_marshal(O.mul(BN, 0xC0FFEE + seed, (1, 2)))
    pts = bytearray(loader.bn254_point_chain(G, step, n))
    if with_infinity:
        for i in range(3, n, 97):
            pts[64 * i:64 * i + 64] = bytes(64)
    sc = b"".join(hashlib.sha256(b"multi%d" % seed + i.to_bytes(4, "little")).digest() for i in range(n))
    return bytes(pts), sc


@pytest.fixture(autouse=True)
def _oversubscribe(monkeypatch):
    monkeypatch.setenv("PORLA_OVERSUBSCRIBE_DEVICES", "1")


@pytest.mark.parametrize("n,ndev", [(1, 2), (7, 3), (4999, 3), (20000, 4), (70001, 8)])
def test_sharded_table_matches_oracle(n, ndev):
    pts, sc = _inputs(n, n)
    want = loader.bn254_msm(sc, pts, n, 4)
    mt = pb.MultiTable(pb.CURVE_BN254, pts, n, ndev=min(ndev, 16))
    assert mt.ndev == ndev
    covered = 0
    for p in range(mt.ndev):
        dev, first, count = mt.part_range(p)
        assert first == covered and 0 <= dev < max(1, pb.load().porla_device_count())
        covered += count
    assert covered == n
    assert mt.msm_host_scalars(sc) == want
    ptrs = mt.upload_scalars(sc)
    assert mt.msm_resident(ptrs) == want
    assert mt.msm_resident(ptrs) == want          # the per-device buffers are reusable
    mt.free_scalars(ptrs)
    mt.destroy()


@pytest.mark.parametrize("curve", [pb.CURVE_BN254, pb.CURVE_SECP256K1])
def test_host_buffer_fanout_matches_single_device(curve):
    """porla_msm_host_devices over 1, 2, 3 and 5 parts returns the bytes of the single-device call (and of the oracle)."""
    n = 30011
    if curve == pb.CURVE_BN254:
        pts, sc = _inputs(n, 5)
        fmt = pb.SCALAR_BE32
        want = loader.bn254_msm(sc, pts, n, 4)
    else:
        c = O.SECP256K1
        rnd = random.Random(9)
        Q = O.mul(c, 0x1234567, (c.gx, c.gy))
        cur, plist = (c.gx, c.gy), []
        for _ in range(n):
            plist.append(cur)
            cur = O.add(c, cur, Q)
        pts = b"".join(P[0].to_bytes(32, "big") + P[1].to_bytes(32, "big") for P in plist)
        sl = [rnd.randrange(1 << 256) for _ in range(n)]
        sc = b"".join(s.to_bytes(32, "little") for s in sl)
        fmt = pb.SCALAR_LE32
        want = pb.msm_host(curve, sc, pts, n, scalar_fmt=fmt)
    for ndev in (1, 2, 3, 5):
        assert pb.msm_host_devices(curve, sc, pts, n, ndev, scalar_fmt=fmt) == want, ndev


@pytest.mark.parametrize("parts", [2, 3, 8])
@pytest.mark.parametrize("kind", ["uniform", "constant", "small31", "top_bucket", "pairs_cancel"])
def test_streamed_parts_share_one_bucket_set(parts, kind, monkeypatch):
    """msm_host_pipelined: the terms arrive in parts, every part is accumulated INTO the buckets the earlier parts filled and
    the buckets are reduced once.  Forced on small inputs (PORLA_STREAM_PARTS) with the cases that stress the carry-over:
    a constant scalar (one bucket per window, cut by every slice and continued by every part), 31-bit scalars (empty top
    windows), digits of the largest magnitude 2^(c-1) (the last bucket of every window), and points that cancel ACROSS
    parts (P in one part, -P in another: the bucket returns to infinity)."""
    n = 6000
    pts, sc = _inputs(n, 11 + parts)
    if kind == "constant":
        sc = sc[:32] * n
    elif kind == "small31":
        sc = b"".join(bytes(28) + sc[32 * i + 28:32 * i + 32] for i in range(n))
    elif kind == "top_bucket":
        # digits of magnitude 2^(c-1) for every window size between 8 and 20, mixed with random scalars
        pats = [sum(1 << (c * w + c - 1) for w in range(0, 250 // c)) for c in range(8, 21)]
        sc = b"".join((pats[i % len(pats)] if i % 3 else int.from_bytes(sc[32 * i:32 * i + 32], "big")).to_bytes(32, "big")
                      for i in range(n))
    elif kind == "pairs_cancel":
        half = n // 2
        P = bytearray(pts)
        neg = bytearray()
        for i in range(half):
            x, y = pts[64 * i:64 * i + 32], int.from_bytes(pts[64 * i + 32:64 * i + 64], "big")
            neg += x + ((BN.p - y) % BN.p if y else 0).to_bytes(32, "big")
        P[64 * half:64 * n] = neg[:64 * (n - half)]
        pts = bytes(P)
        sc = sc[:32 * half] + sc[:32 * (n - half)]          # term i + half = -(term i), except the first few made different
        sc = sc[:32 * half] + bytes(31) + b"\x05" + sc[32 * (half + 1):]
    want = loader.bn254_msm(sc, pts, n, 4)
    monkeypatch.setenv("PORLA_STREAM_PARTS", str(parts))
    assert pb.msm_host_devices(pb.CURVE_BN254, sc, pts, n, 1) == want
    assert pb.msm_host_devices(pb.CURVE_BN254, sc, pts, n, 2) == want      # two devices (or two workers), each streaming its range
    mt = pb.MultiTable(pb.CURVE_BN254, pts, n, ndev=2)                     # resident sharded table, host scalars streamed in parts
    assert mt.msm_host_scalars(sc) == want
    mt.destroy()
    monkeypatch.setenv("PORLA_NO_GLV", "1")
    assert pb.msm_host_devices(pb.CURVE_BN254, sc, pts, n, 1) == want


def test_pageable_buffers_go_through_the_copy_ring():
    """The host-buffer MSM with ordinary heap buffers (what utils.h:277-292 passes): large pageable buffers reach the device
    through the pinned ring of the copy pool, the result is that of the oracle; pinned buffers bypass the ring."""
    import torch
    lib = pb.load()
    n = 1 << 17
    pts, sc = _inputs(n, 77)
    want = loader.bn254_msm(sc, pts, n, 8)
    b_sc, b_pt = bytearray(sc), bytearray(pts)                          # bytearrays: pageable
    before = lib.porla_debug_copy_ring_bytes()
    assert pb.msm_host_devices(pb.CURVE_BN254, b_sc, b_pt, n, 1) == want
    assert lib.porla_debug_copy_ring_bytes() - before == n * 96
    h_sc = torch.frombuffer(bytearray(sc), dtype=torch.uint8).pin_memory()
    h_pt = torch.frombuffer(bytearray(pts), dtype=torch.uint8).pin_memory()
    before = lib.porla_debug_copy_ring_bytes()
    assert pb.msm_host_devices(pb.CURVE_BN254, h_sc.data_ptr(), h_pt.data_ptr(), n, 1) == want
    assert lib.porla_debug_copy_ring_bytes() == before
    # the legacy symbol over the same pageable buffers
    assert pb.bn254_multi_exp(pts, sc, n) == want


def _closed_form_inputs(torch, n, lo, hi, a, b, device):
    """Points (i + 1) G and scalars a i + b for i in [lo, hi) on `device` (tests/test_gpu_fullsize.py's closed form)."""
    from tests.test_gpu_fullsize import _limbs_of
    i = torch.arange(lo, hi, dtype=torch.int64, device=device)
    ks = torch.zeros((hi - lo, 8), dtype=torch.int32, device=device)
    ks[:, 0] = (i + 1).to(torch.int32)
    ss = torch.empty((hi - lo, 8), dtype=torch.int32, device=device)
    carry = torch.zeros(hi - lo, dtype=torch.int64, device=device)
    for j, (al, bl) in enumerate(zip(_limbs_of(a), _limbs_of(b))):
        v = i * al + bl + carry
        lo32 = v & 0xFFFFFFFF
        carry = v >> 32
        ss[:, j] = (lo32 - ((lo32 >> 31) << 32)).to(torch.int32)
    return ks, ss


def _closed_form_bytes(n, a, b):
    total = (a * ((n - 1) * n * (n + 1) // 3) + b * (n * (n + 1) // 2)) % BN.n
    return O.bn254_marshal(O.mul(BN, total, (1, 2)))


def test_two_real_devices_closed_form():
    """2^20 terms over two physical GPUs inside one process: sharded resident table and host-buffer fan-out."""
    import torch
    lib = pb.load()
    if lib.porla_device_count() < 2:
        pytest.skip("needs two CUDA devices")
    n = 1 << 20
    rnd = random.Random(4)
    a = rnd.getrandbits(228) | (1 << 227) | 1
    b = rnd.getrandbits(255) | (1 << 254)
    ks, ss = _closed_form_inputs(torch, n, 0, n, a, b, "cuda:0")
    tab = pb.Table.multiples_of_generator(pb.CURVE_BN254, ks.data_ptr(), n, pb.SCALAR_LE32, on_device=True)
    pts = tab.export()
    tab.destroy()
    sc = ss.cpu().numpy().tobytes()
    want = _closed_form_bytes(n, a, b)
    for ndev in (2, lib.porla_device_count()):
        mt = pb.MultiTable(pb.CURVE_BN254, pts, n, ndev=ndev)
        devs = {mt.part_range(p)[0] for p in range(mt.ndev)}
        assert len(devs) == min(ndev, lib.porla_device_count())
        assert mt.msm_host_scalars(sc, scalar_fmt=pb.SCALAR_LE32) == want
        mt.destroy()
        assert pb.msm_host_devices(pb.CURVE_BN254, sc, pts, n, ndev, scalar_fmt=pb.SCALAR_LE32) == want


def _nccl_worker(rank, world, port, log2n, a, b, q):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["PORLA_DEVICE"] = str(rank)
    import torch
    import torch.distributed as dist
    import porla_b200 as pb2
    from porla_b200.sharding import ShardedMsm, shard_range
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    n = 1 << log2n
    lo, hi = shard_range(n, world, rank)
    ks, ss = _closed_form_inputs(torch, n, lo, hi, a, b, "cuda:%d" % rank)
    tab = pb2.Table.multiples_of_generator(pb2.CURVE_BN254, ks.data_ptr(), hi - lo, pb2.SCALAR_LE32, on_device=True)
    eng = ShardedMsm(pb2.CURVE_BN254, n, world, rank, dist, torch.device("cuda", rank))
    got = eng.msm(tab, ss.data_ptr(), hi - lo, pb2.SCALAR_LE32)
    if rank == 0:
        q.put(got.hex())
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_nccl_sharded_msm_closed_form():
    """One process per GPU (the torchrun layout of bench.py): every rank runs the real CUDA pipeline over its point range,
    the per-window sums meet in one NCCL all-gather, rank 0 combines; the result is the closed form."""
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    log2n, world = 19, 2
    rnd = random.Random(8)
    a = rnd.getrandbits(228) | (1 << 227) | 1
    b = rnd.getrandbits(255) | (1 << 254)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, log2n, a, b, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = q.get(timeout=300)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert got == _closed_form_bytes(1 << log2n, a, b).hex()


def test_fixed_base_window_sums_add_up_on_one_device():
    """PORLA_PLAN_FIXED: two range shards whose tables carry the fixed-base expansion with the same window size contribute
    one XYZZ sum each; combined with nwin = 1 they give the MSM.  A table without the expansion is refused upstream
    (the call aborts), so only the accepted form is exercised here."""
    import torch
    lib = pb.load()
    n, c = 60000, 14
    pts, sc = _inputs(n, 123)
    want = loader.bn254_msm(sc, pts, n, 8)
    half = n // 2
    tabs = [pb.Table.from_host(pb.CURVE_BN254, pts[:64 * half]), pb.Table.from_host(pb.CURVE_BN254, pts[64 * half:])]
    for t in tabs:
        assert t.precompute(c, n, 1) == c
    d_sc = torch.frombuffer(bytearray(sc), dtype=torch.uint8).cuda()
    ws = torch.zeros(2 * 128, dtype=torch.uint8, device="cuda")
    code = c | pb.lib.PLAN_FIXED | pb.lib.PLAN_GLV_OFF
    lib.porla_msm_window_sums_device(C.c_void_p(tabs[0].handle), C.c_void_p(d_sc.data_ptr()), half, pb.SCALAR_BE32, code,
                                     C.c_void_p(ws.data_ptr()), None)
    lib.porla_msm_window_sums_device(C.c_void_p(tabs[1].handle), C.c_void_p(d_sc.data_ptr() + 32 * half), n - half, pb.SCALAR_BE32, code,
                                     C.c_void_p(ws.data_ptr() + 128), None)
    torch.cuda.synchronize()
    out = (C.c_ubyte * 64)()
    lib.porla_msm_finalize_host(pb.CURVE_BN254, ws.cpu().numpy().tobytes(), 2, 1, code, pb.POINT_BE64, C.cast(out, C.c_void_p))
    assert bytes(out) == want
    for t in tabs:
        t.destroy()
