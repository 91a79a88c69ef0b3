"""One-process-per-GPU plumbing around libogb's multi-rank contexts (torch.distributed only moves the
NCCL unique id and the timing scalars; the data-path collectives -- allgather of the index slices, of the packed pre-reduction
adjacency, flags and final edges -- are NCCL calls inside libogb, see csrc/ogb_device.cu)."""
import os

import torch
import torch.distributed as dist


def env_rank():
    """(rank, world_size, local_rank) from the torchrun environment (1 process: 0, 1, 0)."""
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


def shard_bounds(n, rank, world):
    """Query-read shard [lo, hi) of `rank`: contiguous ID ranges of ceil(n/world) reads -- the same rule
    as ogb_context::shard() in csrc/ogb_device.cu (read IDs are lexicographic ranks, i.e. effectively
    random with respect to genome position, so equal ranges carry equal work)."""
    per = (n + world - 1) // world
    return min(n, per * rank), min(n, per * (rank + 1))


def unitig_range(edges, rank, world, canonical=True):
    """(first, count) of the unitigs `rank` spells (OverlapGraph.spell / unitigs) given the simplified graph's edges
    (OverlapGraph.simplify()): the contiguous ranges of shard_bounds over the selected edges. Every rank holds the whole simplified
    graph, so the split needs no collective."""
    import numpy as np
    n = len(edges)
    if canonical:
        i = np.arange(n)
        n = int(((edges["src"] < edges["dst"]) | ((edges["src"] == edges["dst"]) & (i < edges["twin"]))).sum())
    lo, hi = shard_bounds(n, rank, world)
    return lo, hi - lo


def broadcast_bytes(payload, src=0):
    """Broadcasts a bytes object made on `src` (the 128-byte ncclUniqueId) to every rank."""
    box = [payload if dist.get_rank() == src else None]
    dist.broadcast_object_list(box, src=src)
    return box[0]


def max_over_ranks(values, device="cpu"):
    """Element-wise max over ranks of a list of floats (per-step device times)."""
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.cpu().tolist()


def make_context(backend="nccl"):
    """Initialises torch.distributed (when WORLD_SIZE > 1) and returns (Context, rank, world, local_rank)."""
    from .api import Context, nccl_unique_id
    rank, world, local = env_rank()
    uid = None
    if backend == "nccl" and torch.cuda.is_available():
        torch.cuda.set_device(local)      # object collectives stage through the current device
    if world > 1:
        if not dist.is_initialized():
            kw = {"device_id": torch.device("cuda", local)} if backend == "nccl" else {}
            dist.init_process_group(backend, **kw)
        uid = broadcast_bytes(nccl_unique_id() if rank == 0 else None)
    return Context(local, rank, world, uid), rank, world, local


def shared_packed_reads(make_dataset, rank, world, tag="ogb"):
    """One Dataset stage per node instead of one per rank: rank 0 calls make_dataset() -> Dataset, the packed reads reach the
    other ranks' hosts through /dev/shm (memory-mapped, not copied). Returns (words, word_offsets, lengths, meta) with
    meta = dict(n, uniform, L): word_offsets / lengths are None on ranks > 0 for one read length (they are implied)."""
    import numpy as np
    base = f"/dev/shm/{tag}_{os.environ.get('MASTER_PORT', '0')}_{os.getppid() if world > 1 else os.getpid()}"
    meta, words, woffs, lens = None, None, None, None
    if rank == 0:
        ds = make_dataset()
        words, woffs, lens = ds.packed()
        uniform = len(lens) > 0 and int(lens.min()) == int(lens.max())
        meta = dict(n=len(lens), uniform=bool(uniform), L=int(lens[0]) if uniform else 0)
        if world > 1:
            np.save(base + "_words.npy", words)
            if not uniform:
                np.save(base + "_woffs.npy", woffs)
                np.save(base + "_lens.npy", lens)
        words, woffs, lens = np.array(words), np.array(woffs), np.array(lens)      # own copies: the Dataset may go away
    if world > 1:
        meta = broadcast_bytes(meta)
        if rank != 0:
            words = np.load(base + "_words.npy", mmap_mode="r")
            if not meta["uniform"]:
                woffs, lens = np.load(base + "_woffs.npy", mmap_mode="r"), np.load(base + "_lens.npy", mmap_mode="r")
        dist.barrier()
        if rank == 0:
            for suffix in ("_words.npy", "_woffs.npy", "_lens.npy"):
                if os.path.exists(base + suffix):
                    os.remove(base + suffix)           # the mappings of the other ranks stay valid
    return words, woffs, lens, meta


def upload_shared(ctx, words, woffs, lens, meta, rank, world):
    """Replicates the packed reads in every rank's HBM: one read length -> every rank uploads its own shard and the shards are
    allgathered over NVLink (ogb_reads_upload_packed_sharded); mixed lengths -> every rank uploads everything."""
    import numpy as np
    from ._lib import check, lib
    n = meta["n"]
    if meta["uniform"] and world > 1:
        nw = (meta["L"] + 31) // 32
        lo, hi = shard_bounds(n, rank, world)
        mine = np.ascontiguousarray(words[lo * nw:hi * nw])
        check(lib().ogb_reads_upload_packed_sharded(ctx._h, mine.ctypes.data, n, meta["L"]))
    else:
        w, o, l = np.ascontiguousarray(words), np.ascontiguousarray(woffs), np.ascontiguousarray(lens)
        check(lib().ogb_reads_upload_packed(ctx._h, w.ctypes.data, o.ctypes.data, l.ctypes.data, n))
