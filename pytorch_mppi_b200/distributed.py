"""K-sharding across the GPUs of one NVSwitch box (SURVEY.md §8e).

Samples are independent until the softmin, so rank g rolls out the contiguous slice
[k_offset, k_offset + K_local) of the GLOBAL sample index space.  Philox is keyed by the global
index, so the union of all shards is the same sample set for any world size.  Per command each rank
contributes one record (beta_g, eta_g, V_g[R]) of (2+R) doubles:

* exchange="p2p"  : the kernel's finisher stores the record straight into every peer's mailbox
                    over NVLink (8-byte flagged words, LL style) and spins on its own mailbox — no
                    second launch, no NCCL call on the hot path.
* exchange="nccl" : the kernel exports the record, `all_gather_into_tensor` moves it, and
                    `mppi_apply_partials` finishes the update.

Every rank then applies the identical combination in fixed rank order, so U stays bit-identical
across ranks without a broadcast.
"""
from __future__ import annotations

import ctypes as C

import torch


def shard_bounds(K: int, rank: int, world: int):
    """(k_offset, K_local) of `rank`'s contiguous slice; the first K % world ranks get one extra."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, rem = divmod(K, world)
    k_local = base + (1 if rank < rem else 0)
    k_off = rank * base + min(rank, rem)
    if k_local < 1:
        raise ValueError(f"K={K} is smaller than the world size {world}")
    return k_off, k_local


def combine_partials(records: torch.Tensor, lambda_: float):
    """Host-side statement of the cross-rank combination the kernels perform (used by the gloo
    tests): records (G, 2+R) float64 -> (beta, eta, delta (R,)) with
    beta=min beta_g, s_g=exp(-(beta_g-beta)/lambda), eta=sum s_g eta_g, delta=sum s_g V_g / eta."""
    beta = records[:, 0].min()
    s = torch.exp(-(1.0 / lambda_) * (records[:, 0] - beta))
    eta = (s * records[:, 1]).sum()
    delta = (s[:, None] * records[:, 2:]).sum(dim=0) / eta
    return beta, eta, delta


class PeerMailboxes:
    """One small cudaMalloc'd mailbox per rank, mapped into every peer through CUDA IPC."""

    def __init__(self, lib, group, device):
        import torch.distributed as dist
        self.lib = lib
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        from . import _cabi
        with torch.cuda.device(device):
            own = C.c_void_p()
            handle = (C.c_ubyte * 64)()
            _cabi.check(lib.mppi_xchg_create(C.byref(own), handle), "mppi_xchg_create")
            self.own = own.value
            handles = [None] * self.world
            dist.all_gather_object(handles, bytes(handle), group=group)
            self.ptrs = []
            self._opened = []
            for g in range(self.world):
                if g == self.rank:
                    self.ptrs.append(self.own)
                    continue
                peer = C.c_void_p()
                buf = (C.c_ubyte * 64).from_buffer_copy(handles[g])
                _cabi.check(lib.mppi_xchg_open(buf, C.byref(peer)), "mppi_xchg_open")
                self.ptrs.append(peer.value)
                self._opened.append(peer.value)
            dist.barrier(group=group)

    def close(self):
        for ptr in self._opened:
            self.lib.mppi_xchg_close(ptr)
        self._opened = []
        if self.own:
            self.lib.mppi_xchg_destroy(self.own)
            self.own = None
