"""Host-side logic of the range-sharded MSM (SURVEY.md 8(e)): which points a rank owns and how the
per-rank window sums are exchanged and combined.  The reference's analogue is the 8-way contiguous
range partition of /root/reference/porla/Client/Client.hpp:747-787 (thread t owns
[t*n/8, (t+1)*n/8), partial sums added serially); here the partition is over GPUs/processes and
the exchange is one all-gather of nwin*128 bytes per rank (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from typing import Tuple


def shard_range(n: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous range [lo, hi) of rank `rank`; the last rank takes the remainder, exactly as
    Client.hpp:753-754 gives the last thread `n_points - n_point_each_thread*t`."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError("bad world/rank")
    each = n // world
    lo = each * rank
    hi = n if rank == world - 1 else lo + each
    return lo, hi


def gather_window_sums(local, world: int, dist=None):
    """All-gather the per-rank window-sum buffer (a torch.uint8 tensor of nwin*128 bytes).
    Returns a tensor of world*nwin*128 bytes ordered by rank.  `dist` defaults to
    torch.distributed; with world == 1 nothing is exchanged."""
    if world == 1:
        return local
    import torch
    if dist is None:
        import torch.distributed as dist  # type: ignore
    out = torch.empty(local.numel() * world, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local)
    return out


class ShardedMsm:
    """One MSM of `n_total` terms over `world` processes, one GPU each (the torchrun layout; SURVEY.md 8(e)): rank r holds
    the points of shard_range(n_total, world, r) resident in its own HBM.  Every call runs the CUDA pipeline over the
    local range up to the per-window sums, exchanges them in ONE all-gather (nwin * 128 bytes per rank, the only
    data-path collective) and combines on rank 0: parts added window by window, Horner over the windows, normalise.
    All ranks use the window layout planned for the LARGEST shard, so their window sums are addable."""

    def __init__(self, curve: int, n_total: int, world: int, rank: int, dist, device, fixed_base_bits: int = 0):
        """fixed_base_bits = c > 0: the table is a fixed base (an SRS) and every rank has expanded its range with
        table.precompute(c) -- all windows share one bucket set, a rank contributes ONE partial sum (PORLA_PLAN_FIXED)."""
        import ctypes as C
        import torch
        from . import lib as L
        self.C, self.torch, self.L = C, torch, L
        self.lib = L.load()
        self.curve, self.world, self.rank, self.dist = curve, world, rank, dist
        largest = n_total - (n_total // world) * (world - 1)
        c_, w_ = C.c_int(0), C.c_int(0)
        self.lib.porla_msm_plan(curve, largest, 1, 0, C.byref(c_), C.byref(w_))
        self.plan_code, self.nwin = c_.value, w_.value
        if fixed_base_bits > 0:
            self.plan_code, self.nwin = fixed_base_bits | L.PLAN_FIXED | L.PLAN_GLV_OFF, 1
        self.wsum = torch.zeros(self.nwin * 128, dtype=torch.uint8, device=device)
        self.host = torch.zeros(world * self.nwin * 128, dtype=torch.uint8)
        if torch.cuda.is_available():        # (the CPU tests build the engine for its plan only)
            self.host = self.host.pin_memory()
        self.out = (C.c_ubyte * 64)()

    def msm(self, table, d_scalars: int, n_local: int, scalar_fmt: int, out_fmt: int = 0, stream: int = 0):
        """Returns the 64-byte result on rank 0, None on the other ranks."""
        C = self.C
        if stream == 0:
            stream = self.torch.cuda.current_stream().cuda_stream
        self.lib.porla_msm_window_sums_device(C.c_void_p(table.handle), C.c_void_p(d_scalars), n_local, scalar_fmt, self.plan_code,
                                              C.c_void_p(self.wsum.data_ptr()), C.c_void_p(stream))
        allw = gather_window_sums(self.wsum, self.world, self.dist)
        if self.rank != 0:
            return None
        self.host.copy_(allw, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()
        self.lib.porla_msm_finalize_host(self.curve, C.c_void_p(self.host.data_ptr()), self.world, self.nwin, self.plan_code, out_fmt,
                                         C.cast(self.out, C.c_void_p))
        return bytes(self.out)

