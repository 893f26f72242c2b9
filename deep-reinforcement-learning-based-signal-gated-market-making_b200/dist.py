"""Population sharding across the GPUs of one box (SURVEY.md 8e).

The path shards by contiguous global index: rank r evaluates children [first, first+count) of
the SAME (master, sigma, seed, generation) -- children are regenerated from the counter-based
stream, so no genome ever crosses NVLink.  Per generation the only exchange is ONE all-gather of
each rank's packed block (fitness f64 + trade counts i32), after which every rank runs the identical
argmax / tell / validate / select locally.  Works with any torch.distributed backend (NCCL on
the B200 box, gloo in the CPU tests).
"""
from __future__ import annotations

import torch
import torch.distributed as dist


def shard_bounds(pop_size: int, world_size: int, rank: int):
    """Equal contiguous shards of ``stride = ceil(P/R)``; the last ranks may be short or empty."""
    stride = (pop_size + world_size - 1) // world_size
    first = min(rank * stride, pop_size)
    count = min(stride, pop_size - first)
    return first, count, stride


def all_gather_slices(local: torch.Tensor, pop_size: int, stride: int, fill, group=None) -> torch.Tensor:
    """All-gather per-rank slices (padded to ``stride``) and return the first ``pop_size``
    entries in global-index order."""
    world = dist.get_world_size(group)
    padded = torch.full((stride,), fill, dtype=local.dtype, device=local.device)
    padded[:local.numel()] = local
    out = torch.empty(world * stride, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded, group=group)
    return out[:pop_size]


def device_tensor(ptr: int, n: int, dtype: torch.dtype, device: int) -> torch.Tensor:
    """Zero-copy torch view of a raw device buffer owned by the C library."""
    class _Raw:
        pass
    r = _Raw()
    typestr = {torch.float64: "<f8", torch.int32: "<i4", torch.float32: "<f4", torch.uint8: "|u1"}[dtype]
    r.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (int(ptr), False), "version": 2}
    return torch.as_tensor(r, device=f"cuda:{device}")


def block_layout(stride: int):
    """Byte layout of one rank's block of the gather buffer (include/sgmm.h, sgmm_ga_buffers):
    ``fitness f64[stride] | trades i32[stride] | pad to 16 B``.  Returns ``(block_bytes, trades_offset)``."""
    return (stride * 12 + 15) // 16 * 16, stride * 8


def pack_block(fit, trd, stride: int) -> torch.Tensor:
    """Host-side twin of the library's block (used by the gloo tests and by callers that evaluate on their own):
    uint8[block_bytes] holding this rank's fitness and trade slices, zero padded."""
    nbytes, off = block_layout(stride)
    buf = torch.zeros(nbytes, dtype=torch.uint8)
    f = torch.as_tensor(fit, dtype=torch.float64).contiguous()
    t = torch.as_tensor(trd, dtype=torch.int32).contiguous()
    buf[:f.numel() * 8] = f.view(torch.uint8)
    buf[off:off + t.numel() * 4] = t.view(torch.uint8)
    return buf


def unpack_blocks(buf: torch.Tensor, world: int, stride: int, pop_size: int):
    """Inverse of :func:`pack_block` over the gathered buffer: ``(fitness f64[pop], trades i32[pop])`` in global order."""
    nbytes, off = block_layout(stride)
    b = buf.reshape(world, nbytes)
    fit = b[:, :stride * 8].contiguous().view(torch.float64).reshape(-1)[:pop_size]
    trd = b[:, off:off + stride * 4].contiguous().view(torch.int32).reshape(-1)[:pop_size]
    return fit, trd


def all_gather_packed(fit, trd, pop_size: int, stride: int, group=None):
    """ONE all-gather per generation: every rank contributes its packed (fitness, trades) block."""
    world = dist.get_world_size(group)
    mine = pack_block(fit, trd, stride)
    out = torch.empty(world * mine.numel(), dtype=torch.uint8)
    dist.all_gather_into_tensor(out, mine, group=group)
    return unpack_blocks(out, world, stride, pop_size)


class ShardedGA:
    """One process per GPU: evaluate the local shard, ONE in-place all-gather of this rank's (fitness, trades) block
    into the library's rank-blocked gather buffer, select locally (identical on every rank).  Replaces the
    ``Pool.starmap`` fan-out / result list of Env/drl_engine.py:104-125 across the GPUs of one box.

    ``objective`` (``"reward"``, ``"pnl"``, ``"pnl_map"``, ``"sharpe"``; None = whatever ``make_ga`` set) is set on the
    rank's GA before its first generation (``sgmm_ga_set_objective``).  Every rank must pass the same one; the objective
    is per child, so the exchange is unchanged."""

    def __init__(self, make_ga, pop_size, group=None, objective=None):
        self.group = group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.pop_size = pop_size
        self.first, self.count, self.stride = shard_bounds(pop_size, self.world, self.rank)
        self.ga = make_ga((self.first, self.count, self.stride))
        if objective is not None:
            self.ga.set_objective(objective)
        _, _, base, block_bytes, n_blocks, my_block = self.ga.buffers()
        assert n_blocks <= self.world and block_bytes == block_layout(self.stride)[0]
        dev = self.ga.device
        # the library allocates n_blocks = ceil(P / stride) blocks; ranks beyond that own an empty shard and contribute
        # (and receive) nothing meaningful -- the collective still needs world blocks, so gather into a private buffer then
        self._direct = (n_blocks == self.world)
        if self._direct:
            self.gather = device_tensor(base, self.world * block_bytes, torch.uint8, dev)
        else:
            self.gather = torch.zeros(self.world * block_bytes, dtype=torch.uint8, device=f"cuda:{dev}")
            self._lib_view = device_tensor(base, n_blocks * block_bytes, torch.uint8, dev)
        self.block_bytes, self.n_blocks, self.my_block = block_bytes, n_blocks, my_block
        self.mine = self.gather[self.rank * block_bytes:(self.rank + 1) * block_bytes]
        self.collectives = 0

    def exchange(self):
        if self.world == 1:
            return
        if not self._direct and self.rank < self.n_blocks:
            self.mine.copy_(self._lib_view[self.rank * self.block_bytes:(self.rank + 1) * self.block_bytes])
        dist.all_gather_into_tensor(self.gather, self.mine, group=self.group)
        self.collectives += 1
        if not self._direct:
            self._lib_view.copy_(self.gather[:self.n_blocks * self.block_bytes])

    def generation(self, train, val):
        self.ga.evaluate(train)
        self.exchange()
        self.ga.select(val)
