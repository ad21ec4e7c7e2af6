"""Multi-GPU modes of the mapping path (SURVEY.md 8e).

Mode 1, read sharding: reads are independent (sigmap.cc:630-866 touches only its own read and
the read-only index), so ranks map disjoint slices of the read set against a replicated index and
the only exchange is the final gather of the fixed-size result rows.  No data-path collective.
Works on any torch.distributed backend (nccl on the GPU box, gloo in the CPU tests).

Mode 2, contig-sharded index (references whose index exceeds one GPU): contigs are bin-packed
over the ranks (`assign_contigs`), every rank maps every read against its own contigs, and the
library's three small collectives per pipeline step (sb_exchange.cuh) make every rank return the
rows of the unsharded run.  `nccl_join` sets this up for one-process-per-GPU runs (NCCL over
NVLink, unique id broadcast through torch.distributed); `ContigShardGroup` does the same for
several contexts inside one process (one host thread per context), which is how the path is
parity-tested on a single GPU.
"""
import ctypes as C

import numpy as np


def block_range(n_items, world, rank):
    """Contiguous, balanced slice [lo, hi) of n_items owned by `rank` (first n % world ranks get
    one extra item).  Concatenating the slices in rank order restores the original order."""
    base, extra = divmod(int(n_items), int(world))
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def shard_reads(reads, world, rank):
    """The ReadSet slice of this rank (views into the same raw buffer; offsets rebased)."""
    from .host import ReadSet
    lo, hi = block_range(reads.n, world, rank)
    s0, s1 = int(reads.read_off[lo]), int(reads.read_off[hi])
    sub = ReadSet(reads.names[lo:hi], reads.raw[s0:s1], reads.read_off[lo:hi + 1] - np.uint64(s0),
                  1.0, 1.0, 0.0, None if reads.truth is None else reads.truth[lo:hi])
    sub.digitisation = reads.digitisation[lo:hi].copy()
    sub.range = reads.range[lo:hi].copy()
    sub.offset = reads.offset[lo:hi].copy()
    return sub


def rows_to_array(rows, struct_type):
    """list of ctypes structs -> uint8 array (n, sizeof)"""
    size = C.sizeof(struct_type)
    out = np.zeros((len(rows), size), np.uint8)
    for i, r in enumerate(rows):
        out[i] = np.frombuffer(bytes(r), np.uint8)
    return out


def array_to_rows(arr, struct_type):
    return [struct_type.from_buffer_copy(arr[i].tobytes()) for i in range(arr.shape[0])]


def gather_rows(rows, struct_type, dist=None, device="cpu"):
    """Every rank contributes its result rows (ctypes structs); rank 0 returns all rows in rank
    order (= read order under block_range sharding), other ranks return None."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return list(rows)
    import torch
    world, rank = dist.get_world_size(), dist.get_rank()
    mine = torch.from_numpy(rows_to_array(rows, struct_type)).to(device)
    counts = [torch.zeros(1, dtype=torch.int64, device=device) for _ in range(world)]
    dist.all_gather(counts, torch.tensor([mine.shape[0]], dtype=torch.int64, device=device))
    counts = [int(c.item()) for c in counts]
    width = C.sizeof(struct_type)
    padded = torch.zeros((max(counts + [1]), width), dtype=torch.uint8, device=device)
    padded[:mine.shape[0]] = mine
    bufs = [torch.zeros_like(padded) for _ in range(world)]
    dist.all_gather(bufs, padded)
    if rank != 0:
        return None
    out = []
    for r in range(world):
        out.extend(array_to_rows(bufs[r][:counts[r]].cpu().numpy(), struct_type))
    return out


def reduce_scalar(x, op, dist=None, device="cpu"):
    """max / sum of a Python float over ranks (timing is the max over ranks, work the sum)."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return float(x)
    import torch
    t = torch.tensor([float(x)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM)
    return float(t.item())


# ------------------------------------------------------------------ mode 2: contig-sharded index
def assign_contigs(lengths, world):
    """owner[c] = rank holding contig c: longest contigs first onto the lightest rank
    (smbh_assign_contigs; deterministic, so every rank computes the same table)."""
    from . import _ffi as F
    lengths = np.ascontiguousarray(lengths, np.uint32)
    owner = np.zeros(len(lengths), np.uint32)
    rc = F.lib.smbh_assign_contigs(F.ptr(lengths, F.u32p), len(lengths), int(world),
                                   F.ptr(owner, F.u32p))
    if rc != 0:
        raise ValueError("smbh_assign_contigs: world must be >= 1")
    return owner


def nccl_join(mapper, dist):
    """Make `mapper` rank dist.get_rank() of a contig-shard group whose collectives are NCCL calls
    on the mapper's own stream.  The NCCL unique id travels through torch.distributed (any
    backend); afterwards torch is out of the data path."""
    from . import _ffi as F
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [None]
    if rank == 0:
        buf = C.create_string_buffer(128)
        rc = F.lib.smb_shard_nccl_unique_id(buf)
        if rc != 0:
            raise RuntimeError(f"smb_shard_nccl_unique_id failed ({rc}): "
                               f"{F.lib.smb_last_error(None).decode()}")
        box[0] = buf.raw
    dist.broadcast_object_list(box, src=0)
    mapper._check(F.lib.smb_shard_nccl_init(mapper._ctx, rank, world, box[0]), "smb_shard_nccl_init")


class ContigShardGroup:
    """`world` contexts in this process (devices[i] may repeat: shards of one GPU), joined into a
    local shard group.  Collective calls run one host thread per rank."""

    def __init__(self, devices):
        from . import _ffi as F
        from .mapper import Mapper
        self.mappers = [Mapper(d) for d in devices]
        arr = (C.c_void_p * len(self.mappers))(*[m._ctx for m in self.mappers])
        rc = F.lib.smb_shard_local_group(arr, len(self.mappers))
        if rc != 0:
            raise RuntimeError(f"smb_shard_local_group failed ({rc})")

    @property
    def world(self):
        return len(self.mappers)

    def _each(self, fn):
        import threading
        out, err = [None] * self.world, [None] * self.world

        def run(r):
            try:
                out[r] = fn(self.mappers[r])
            except Exception as e:  # noqa: BLE001 - re-raised below
                err[r] = e

        ts = [threading.Thread(target=run, args=(r,)) for r in range(self.world)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        for e in err:
            if e is not None:
                raise e
        return out

    def set_index(self, pos, val, contig_lengths, owner=None):
        owner = assign_contigs(contig_lengths, self.world) if owner is None else owner
        self.owner = np.ascontiguousarray(owner, np.uint32)
        for m in self.mappers:
            m.set_index_sharded(pos, val, self.owner)
            m.set_contigs(contig_lengths)

    def set_index_from_reference(self, ref, level_mean, owner=None):
        """Contig-sharded index where every member builds only ITS OWN part of the point cloud from
        the reference sequences (host.build_point_cloud_part): the way a genome-scale reference is
        indexed, since no member ever holds the whole cloud."""
        from .host import build_point_cloud_part
        owner = assign_contigs(ref.lengths, self.world) if owner is None else owner
        self.owner = np.ascontiguousarray(owner, np.uint32)
        for r, m in enumerate(self.mappers):
            part = build_point_cloud_part(ref, level_mean, self.owner, r)
            try:
                m.set_index_part(part, ref.n)
            finally:
                part.close()
            m.set_contigs(ref.lengths)

    def build_index(self, ref, level_mean, owner=None):
        """Contig-sharded index built on the devices from the reference sequences
        (smb_index_build): each member builds the cloud on its GPU and keeps only its own part."""
        owner = assign_contigs(ref.lengths, self.world) if owner is None else owner
        self.owner = np.ascontiguousarray(owner, np.uint32)
        self._each(lambda m: m.build_index(ref, level_mean, self.owner))

    def replicate_index(self, pos, val, contig_lengths, root=0):
        """Read-sharded mode: the index is built on `root` only and broadcast to the other members
        over NVLink / peer copies (smb_index_broadcast); every member then maps its own reads."""
        self.mappers[root].set_index(pos, val)
        self.mappers[root].set_contigs(contig_lengths)
        self._each(lambda m: m.broadcast_index(root))
        for m in self.mappers:
            m.set_contigs(contig_lengths)

    def map_reads(self, reads, params=None):
        """rows of every rank (list of lists); they are identical by construction."""
        return self._each(lambda m: m.map_reads(reads, params))

    def close(self):
        for m in self.mappers:
            m.close()
