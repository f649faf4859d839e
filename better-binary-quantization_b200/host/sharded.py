"""Row-wise sharded search over the GPUs of one box (SURVEY §8e): one process per GPU, each rank owns a
contiguous row shard (global id = shard base + local row).  The exchange lives IN THE LIBRARY: every rank calls
bbq_search_sharded with the same query batch; the per-shard top-k lists travel as 64-bit (score, id) keys in ONE
ncclAllGather over NVLink (the library dlopens NCCL and owns the communicator) and are merged by the device
selection kernel, so the result is independent of the number of shards.  This file only bootstraps: rank 0 makes
the communicator id (bbq_comm_unique_id) and it is broadcast over whatever the host already has — here
torch.distributed (gloo or nccl), in a Node host a pipe or an environment variable (INTEGRATION.md).
The reference has no counterpart (it is single-process); the merge rule is its MinHeap contract made canonical
(src/binaryQuantizationFormat.ts:383-411).
One process can also drive every GPU itself: BinaryQuantizationFormat(config, devices=[...]) owns a device group
(bbq_group_*), one worker thread per GPU running these same collective entries with the split of shard_bounds below;
no communicator id, rank bookkeeping or corpus split is left to the host."""
from __future__ import annotations

import numpy as np

from .format import BinarizedByteVectorValues, BinaryQuantizationFormat, _index


def shard_bounds(n_total: int, world: int, rank: int):
    """Contiguous shards: rank r owns [r*ceil(n/world), min(n, (r+1)*ceil(n/world)))."""
    per = -(-n_total // world)
    return min(n_total, rank * per), min(n_total, (rank + 1) * per)


def broadcast_comm_id(make_id, rank: int, world: int, group=None) -> bytes:
    """Bootstrap only: rank 0's 128-byte communicator id to every rank through torch.distributed."""
    import torch.distributed as dist
    box = [make_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0, group=group)
    return box[0]


class ShardedSearcher:
    def __init__(self, fmt: BinaryQuantizationFormat, shard: BinarizedByteVectorValues, base: int, rank: int = 0,
                 world: int = 1, group=None):
        import torch
        from .. import _native
        self.torch = torch
        self.fmt, self.shard, self.rank, self.world = fmt, shard, rank, world
        st = _native.load().bbq_index_set_base(_index(shard), int(base))
        if st != 0:
            raise RuntimeError(_native.load().bbq_last_error().decode())
        if world > 1:
            fmt.commInit(broadcast_comm_id(fmt.commUniqueId, rank, world, group), rank, world)
        self.stream = torch.cuda.Stream()
        self._bufs = {}

    def _buffers(self, nq, k, dim):
        key = (nq, k, dim)
        if key not in self._bufs:
            t, dev = self.torch, "cuda"
            self._bufs = {key: dict(
                out_idx=t.empty((nq, k), dtype=t.int32, device=dev),
                out_sc=t.empty((nq, k), dtype=t.float32, device=dev),
                h_idx=t.empty((nq, k), dtype=t.int32, pin_memory=True),
                h_sc=t.empty((nq, k), dtype=t.float32, pin_memory=True))}
        return self._bufs[key]

    def search_device(self, dq, k):
        """dq: [nq, dim] f32 CUDA tensor (replicated on every rank).  Returns (idx, score) CUDA tensors [nq, k];
        enqueued on self.stream (the caller synchronises).  bbq_search_sharded_device: local scan, key pack,
        ncclAllGather, merge — all inside the library."""
        nq, dim = dq.shape
        b = self._buffers(nq, k, dim)
        self.fmt.searchShardedDevice(dq.data_ptr(), nq, self.shard, k, b["out_idx"].data_ptr(), b["out_sc"].data_ptr(),
                                     self.stream.cuda_stream)
        return b["out_idx"], b["out_sc"]

    def search(self, h_queries, k):
        """End-to-end through the entry a host binds: bbq_search_sharded on HOST buffers (h_queries: a CPU tensor,
        pinned for full-speed DMA; pageable works too).  The H2D copy of the queries, the search, the exchange and the
        D2H copy of the results all happen inside the call."""
        nq, dim = h_queries.shape
        b = self._buffers(nq, k, dim)
        cnt = self.fmt.searchShardedHost(h_queries.data_ptr(), nq, self.shard, k, b["h_idx"].data_ptr(),
                                         b["h_sc"].data_ptr())
        return b["h_idx"][:, :cnt], b["h_sc"][:, :cnt]


def merge_host(idx_lists, score_lists, k):
    """Pure-numpy statement of the merge rule (score desc, id asc, empty = id -1) for the gloo CPU tests of the
    multi-rank plumbing; NOT used by the product path."""
    idx = np.concatenate(idx_lists, axis=1)
    sc = np.concatenate(score_lists, axis=1)
    out_i = np.full((idx.shape[0], k), -1, np.int32)
    out_s = np.full((idx.shape[0], k), -np.inf, np.float32)
    for q in range(idx.shape[0]):
        valid = idx[q] >= 0
        i, s = idx[q][valid], sc[q][valid]
        nan = np.isnan(s)
        order = np.lexsort((i, -np.where(nan, -np.inf, s + 0.0), nan))
        order = order[:k]
        out_i[q, :len(order)], out_s[q, :len(order)] = i[order], s[order]
    return out_i, out_s
