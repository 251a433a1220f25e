"""Sharding of the pair list across ranks and the one exchange step of the path.

Scan pairs are independent (SURVEY.md section 8e): every rank holds the whole scan table, aligns
an interleaved-block slice of the problem index space, and an all-gather of fixed-size records
returns every pair's constraint to all ranks (rank 0 feeds the unchanged host-side pose graph).
This replaces the result gather of the reference's joblib fan-out
(``zip(*parallel(...))``, reference scripts/main.py:241).

One process per GPU; ``torch.distributed`` with the nccl backend on GPUs (gloo works for the
host-side logic and is what the CPU tests use).
"""
from __future__ import annotations

import numpy as np

from .icp import _to33, _top_rows, make_epilogue

RECORD_WIDTH = 8     # T (6 doubles), error, passes


def shard_indices(n_problems: int, rank: int, world: int, block: int = 4096) -> np.ndarray:
    """Global problem indices owned by `rank`: blocks rank, rank+world, ... of `block` problems.
    Interleaving evens out the data-dependent pass counts (4..102 per pair)."""
    if not (0 <= rank < world):
        raise ValueError("rank out of range")
    block = max(int(block), 1)
    k = np.arange(n_problems, dtype=np.int64)
    return k[(k // block) % world == rank]


def shard_all_pairs(n_problems: int, rank: int, world: int, block: int = 4096):
    """(k_first, k_block, k_stride, B_local) for the device-decoded all-pairs index space
    (icpb_params pair_mode 1); enumerates exactly shard_indices(...)."""
    block = max(int(block), 1)
    b_local = int(len(shard_indices(n_problems, rank, world, block)))
    return rank * block, block, world * block, b_local


def pack_records(T: np.ndarray, error: np.ndarray, passes: np.ndarray) -> np.ndarray:
    rec = np.empty((len(error), RECORD_WIDTH))
    rec[:, :6] = _top_rows(T)
    rec[:, 6] = error
    rec[:, 7] = passes
    return rec


def unpack_records(rec: np.ndarray):
    return _to33(rec[:, :6]), rec[:, 6].copy(), rec[:, 7].astype(np.int32)


def all_gather_records(local: np.ndarray, n_problems: int, block: int = 4096, group=None, device=None):
    """All-gather per-rank record arrays (rows in shard_indices order) and return the
    (n_problems, 8) array in global problem order on every rank."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    counts = [len(shard_indices(n_problems, r, world, block)) for r in range(world)]
    if len(local) != counts[rank]:
        raise ValueError(f"rank {rank} holds {len(local)} records, expected {counts[rank]}")
    cap = max(counts) if counts else 0
    send = torch.zeros((cap, RECORD_WIDTH), dtype=torch.float64, device=device)
    if len(local):
        send[:len(local)] = torch.from_numpy(np.ascontiguousarray(local)).to(send.device)
    recv = torch.empty((world * cap, RECORD_WIDTH), dtype=torch.float64, device=device)
    dist.all_gather_into_tensor(recv, send, group=group)
    recv = recv.cpu().numpy().reshape(world, cap, RECORD_WIDTH)
    out = np.empty((n_problems, RECORD_WIDTH))
    for r in range(world):
        out[shard_indices(n_problems, r, world, block)] = recv[r, :counts[r]]
    return out


def icp_batch_sharded(align, pairs, init_transforms=None, block: int = 4096, group=None, device=None,
                      **icp_kwargs):
    """Align this rank's slice with `align(pairs, init, **kw) -> BatchResult-like` (normally
    ``IcpEngine.run``) and return (T, error, passes) for ALL pairs on every rank."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    pairs = np.asarray(pairs)
    mine = shard_indices(len(pairs), rank, world, block)
    init = None if init_transforms is None else np.asarray(init_transforms)[mine]
    res = align(pairs[mine], init, **icp_kwargs)
    rec = all_gather_records(pack_records(res.T, res.error, res.iters), len(pairs), block, group, device)
    return unpack_records(rec)


# --------------------------------------------------------------------------- fused gather (NVLink peer memory)
def global_rows(n_problems: int, rank: int, world: int, block: int = 4096):
    """(row0, row_block, row_stride) of icpb_epilogue for `rank`'s interleaved blocks: local problem b
    is global problem row0 + (b // block) * stride + b % block -- exactly shard_indices(...)[b]."""
    block = max(int(block), 1)
    return rank * block, block, world * block


class FusedGather:
    """The exchange step of the sharded path without a collective: every rank's gather buffer lives in
    torch symmetric memory, so each rank has every peer's buffer mapped, and the alignment kernel's
    epilogue stores each finished pair's 64-byte record [T(6), error, passes] straight into ALL of them
    at the pair's GLOBAL row (``icpb_epilogue``, include/icpb.h).  After ``barrier()`` every rank holds
    all ``n_problems`` records in global problem order.  Replaces ``all_gather_records`` (NCCL) and the
    host-side packing in front of it; the reference's counterpart is the result gather of its joblib
    fan-out, ``zip(*parallel(...))`` (scripts/main.py:241).

    With ``accept_cap > 0`` the acceptance test of the loop-closure callers
    (src/loop_closure_detection.py:35-39,155-159) runs in the epilogue too: only pairs with
    error < accept_thresh are appended, into this rank's region of every peer's compact buffer, so
    only accepted constraints cross NVLink.  ``accepted()`` returns them ordered by global problem id.
    """

    def __init__(self, n_problems: int, group=None, device=None, block: int = 4096, accept_cap: int = 0,
                 gather_all: bool = True):
        import torch
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group if group is not None else dist.group.WORLD
        self.world = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        self.n_problems, self.block = int(n_problems), max(int(block), 1)
        self.mine = shard_indices(self.n_problems, self.rank, self.world, self.block)
        self.buf = self.hdl = None
        if gather_all:
            self.buf = symm_mem.empty((max(self.n_problems, 1), RECORD_WIDTH), dtype=torch.float64, device=device)
            self.hdl = symm_mem.rendezvous(self.buf, self.group)
        self.accept_cap = int(accept_cap)
        self.acc = self.acc_hdl = self.cnt = self.cnt_hdl = None
        if self.accept_cap > 0:
            self.acc = symm_mem.empty((self.world * self.accept_cap, RECORD_WIDTH), dtype=torch.float64, device=device)
            self.acc_hdl = symm_mem.rendezvous(self.acc, self.group)
            self.cnt = symm_mem.empty((self.world,), dtype=torch.int64, device=device)
            self.cnt_hdl = symm_mem.rendezvous(self.cnt, self.group)
            self.cnt.zero_()
        self._any = self.hdl or self.acc_hdl

    def epilogue(self, accept_thresh=None):
        row0, rb, rs = global_rows(self.n_problems, self.rank, self.world, self.block)
        kw = {}
        if self.accept_cap > 0 and accept_thresh is not None:
            kw = dict(accept_thresh=accept_thresh, accept_peer_ptrs=int(self.acc_hdl.buffer_ptrs_dev),
                      accept_count_peer_ptrs=int(self.cnt_hdl.buffer_ptrs_dev), accept_cap=self.accept_cap)
        return make_epilogue(int(self.hdl.buffer_ptrs_dev) if self.hdl else 0, self.world, self.rank,
                             row0, rb, rs, **kw)

    def clear(self):
        """Zero the buffers on every rank (tests: stale records must not pass for fresh ones)."""
        if self.buf is not None:
            self.buf.zero_()
        if self.acc is not None:
            self.acc.zero_(); self.cnt.zero_()
        self.barrier()

    def barrier(self):
        """All ranks' launches have completed and their stores have landed everywhere."""
        self._any.barrier()

    def records(self):
        """(n_problems, 8) float64 CUDA tensor, global problem order; valid after barrier()."""
        return self.buf[:self.n_problems]

    def accepted(self):
        """(rows, T (k,3,3), error (k,), passes (k,)) of the accepted pairs, ordered by global problem id;
        valid after barrier().  Raises if a rank overflowed its region."""
        import torch
        cnt = self.cnt.cpu().numpy()
        if (cnt < 0).any():
            raise RuntimeError(f"acceptance buffer overflow (accept_cap {self.accept_cap}, counts {(-cnt).tolist()})")
        parts = [self.acc[r * self.accept_cap:r * self.accept_cap + int(cnt[r])] for r in range(self.world)]
        rec = torch.cat(parts).cpu().numpy() if parts else np.empty((0, RECORD_WIDTH))
        return unpack_accepted(rec)


def unpack_accepted(rec: np.ndarray):
    """Accepted-record rows -> (global problem ids, T, error, passes), sorted by problem id (the
    kernel appends in completion order; the tag in the 8th slot carries (row << 16) | passes)."""
    rec = np.ascontiguousarray(rec, dtype=np.float64).reshape(-1, RECORD_WIDTH)
    tag = rec[:, 7].copy().view(np.int64)
    rows, passes = tag >> 16, (tag & 0xffff).astype(np.int32)
    order = np.argsort(rows, kind="stable")
    return rows[order], _to33(rec[:, :6])[order], rec[order, 6].copy(), passes[order]


def icp_batch_sharded_fused(eng, scans, pairs, init_transforms, gather: FusedGather, accept_thresh=None,
                            **icp_kwargs):
    """The sharded path end to end from host memory: this rank aligns its interleaved slice of `pairs`
    through ``IcpEngine.align`` (upload overlapped with the kernel) with the gather fused into the
    kernel's epilogue, then one symmetric-memory barrier.  Returns (T, error, passes) for ALL pairs on
    every rank, like ``icp_batch_sharded``; with ``accept_thresh`` (and a FusedGather built with
    accept_cap) only the accepted constraints are exchanged and ``gather.accepted()`` has them."""
    pairs = np.asarray(pairs)
    if len(pairs) != gather.n_problems:
        raise ValueError("the FusedGather was sized for a different number of problems")
    mine = gather.mine
    init = None if init_transforms is None else np.asarray(init_transforms)[mine]
    eng.align(scans, pairs[mine], init, epilogue=gather.epilogue(accept_thresh), **icp_kwargs)
    gather.barrier()
    if gather.buf is None:
        return None
    return unpack_records(gather.records().cpu().numpy())
