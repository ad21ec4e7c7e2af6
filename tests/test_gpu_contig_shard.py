"""Contig-sharded index (SURVEY.md 8e mode 2) against the unsharded CUDA path: the contigs of a
multi-contig reference are spread over several shard contexts that live on the one test GPU
(shard.ContigShardGroup: one host thread per rank, in-process exchange), every rank maps every
read, and every rank must return the unsharded run's rows bit for bit -- in the default
(stop-early) mode, in full-read mode where chains are carried over many chunks, and when the
batch has to be split into several pipeline steps.  The unsharded path itself is pinned to the
oracle / reference by test_gpu_parity.py and test_gpu_golden.py."""
import ctypes as C

import numpy as np
import pytest

from conftest import Dataset, paf_cols

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def multi(host, model, tmp_path_factory):
    # 7 contigs of uneven length; noise 1.4 leaves a few reads with several candidate chains
    return Dataset(host, model, tmp_path_factory.mktemp("multi"),
                   [90000, 40000, 120000, 30000, 70000, 55000, 25000], 48, seed=21, noise=1.4,
                   min_bases=1500, max_bases=6000)


@pytest.fixture(scope="module")
def whole(multi):
    from sigmap_b200.mapper import Mapper
    m = Mapper(0)
    m.set_index(multi.pos, multi.val)
    m.set_contigs(multi.ref.lengths)
    yield m
    m.close()


def row_bytes(rows):
    return [bytes(r) for r in rows]


@pytest.fixture(scope="module")
def repeats(host, model):
    from repeat_genome import RepeatGenome
    from sigmap_b200.mapper import Mapper
    g = RepeatGenome(host, model)
    m = Mapper(0)
    m.set_index(g.pos, g.val)
    m.set_contigs(g.ref.lengths)
    yield g, m
    m.close()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_rows_equal_unsharded(multi, whole, repeats, world):
    from sigmap_b200 import shard
    from sigmap_b200.mapper import default_params, full_read_params
    g = shard.ContigShardGroup([0] * world)
    try:
        g.set_index(multi.pos, multi.val, multi.ref.lengths)
        assert sorted(set(g.owner.tolist())) == list(range(world))
        for prm in (default_params(), full_read_params()):
            exp = whole.map_reads(multi.reads, prm)
            got = g.map_reads(multi.reads, prm)
            assert sum(r.mapped for r in exp) > multi.reads.n // 2
            for rank_rows in got:
                assert row_bytes(rank_rows) == row_bytes(exp)
        st = [m.stats() for m in g.mappers]
        assert all(s["exchanges"] > 0 for s in st)
        # every rank searched only its own contigs: the hits add up to the unsharded run's
        whole.stats_reset()
        for m in g.mappers:
            m.stats_reset()
        whole.map_reads(multi.reads, default_params())
        g.map_reads(multi.reads, default_params())
        assert sum(m.stats()["hits"] for m in g.mappers) == whole.stats()["hits"]
        # the repeat genome with B, C and D (exact copies: tied chains) on different ranks, so the
        # tied candidates meet in the exchange and every rank must pick the unsharded winner
        rep, rep_whole = repeats
        owner = [world - 1, 0, 1 % world, 2 % world, 0, 1 % world, 0, world - 1]  # A B C D S t5 t11 t12
        g.set_index(rep.pos, rep.val, rep.ref.lengths, owner=owner)
        for prm in (default_params(), full_read_params()):
            exp = rep_whole.map_reads(rep.reads, prm)
            for rank_rows in g.map_reads(rep.reads, prm):
                assert row_bytes(rank_rows) == row_bytes(exp), "repeats"
    finally:
        g.close()


def test_sharded_split_steps_and_paf(multi, whole):
    """Tiny batch limits force several steps per round and anchor-buffer overflow retries, which
    are collective decisions in a sharded run; the PAF text must still match."""
    from sigmap_b200 import shard
    from sigmap_b200.mapper import full_read_params
    g = shard.ContigShardGroup([0, 0])
    try:
        g.set_index(multi.pos, multi.val, multi.ref.lengths, owner=[0, 1, 0, 1, 0, 1, 1])
        for m in g.mappers:
            m.set_limits(max_batch_chunks=7, max_batch_anchors=60000)
        prm = full_read_params()
        exp = whole.map_reads(multi.reads, prm)
        got = g.map_reads(multi.reads, prm)
        exp_paf = [paf_cols(l) for l in whole.paf_lines(multi.reads, exp, multi.ref.names)]
        for m, rows in zip(g.mappers, got):
            assert [paf_cols(l) for l in m.paf_lines(multi.reads, rows, multi.ref.names)] == exp_paf
    finally:
        g.close()


def test_shard_holds_only_its_contigs(multi, whole, port):
    """Radius-search stage on a shard: exactly the unsharded hits whose point lies on an owned
    contig (same window indices, same d2 bits)."""
    from sigmap_b200 import shard
    g = shard.ContigShardGroup([0, 0])
    try:
        g.set_index(multi.pos, multi.val, multi.ref.lengths)
        f = port.generate_events(multi.pa(port, 0)[:4000])
        q = np.stack([f[p:p + 6] for p in range(2, len(f) - 5, 2)])
        off, idx, d2 = whole.radiusSearch(q)
        contig = (multi.pos[idx.astype(np.int64)] >> np.uint64(33)).astype(np.int64)
        qid = np.repeat(np.arange(len(q)), np.diff(off).astype(np.int64))
        seen = 0
        for r, m in enumerate(g.mappers):
            o2, i2, dd2 = m.radiusSearch(q)
            keep = g.owner[contig] == r
            assert np.array_equal(i2, idx[keep])
            assert np.array_equal(dd2.view(np.uint32), d2[keep].view(np.uint32))
            assert np.array_equal(np.diff(o2).astype(np.int64), np.bincount(qid[keep], minlength=len(q)))
            seen += len(i2)
        assert seen == len(idx) > 0
    finally:
        g.close()


def test_nccl_two_ranks_when_two_gpus():
    """The same check over the NCCL backend, one process per GPU (needs >= 2 GPUs: skipped on the
    single-GPU test box; run with `gpurun --gpus 2`)."""
    import os
    import subprocess
    import sys

    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29517",
                        os.path.join(root, "tools", "shard_nccl_check.py")],
                       capture_output=True, text=True, timeout=600, env=dict(os.environ, CHECK_READS="120"))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "PASS" in r.stdout


def test_broadcast_index_replicas_map_like_the_root(multi, whole):
    """Read-sharded mode: the index built on rank 0 is broadcast to the other members of the group
    (smb_index_broadcast: NCCL across processes, peer copies here); each member then maps its own
    slice of the reads, with no collective on the data path, and the rows are the unsharded run's."""
    from sigmap_b200 import shard
    from sigmap_b200.mapper import default_params
    g = shard.ContigShardGroup([0, 0, 0])
    try:
        g.replicate_index(multi.pos, multi.val, multi.ref.lengths)
        assert all(m.num_points == whole.num_points for m in g.mappers)
        exp = whole.map_reads(multi.reads, default_params())
        for m in g.mappers:
            m.stats_reset()
        parts = [shard.shard_reads(multi.reads, g.world, r) for r in range(g.world)]
        got = g._each(lambda m: m.map_reads(parts[g.mappers.index(m)], default_params()))
        rows = [r for part in got for r in part]
        assert row_bytes(rows) == row_bytes(exp)
        assert all(m.stats()["exchanges"] == 0 for m in g.mappers)  # nothing collective while mapping
    finally:
        g.close()


def test_sharded_index_from_own_cloud_parts(multi, whole, model):
    """The way a genome-scale reference is indexed: every member of the group builds only ITS OWN
    part of the point cloud from the sequences (smbh_build_point_cloud_part) and its device index
    from that (smb_index_set_points_part).  Rows must equal the unsharded run's."""
    from sigmap_b200 import shard
    from sigmap_b200.mapper import default_params, full_read_params
    g = shard.ContigShardGroup([0, 0, 0])
    try:
        g.set_index_from_reference(multi.ref, model[0])
        assert sum(m.stats()["launches"] > 0 for m in g.mappers) == 3
        for prm in (default_params(), full_read_params()):
            exp = whole.map_reads(multi.reads, prm)
            for rank_rows in g.map_reads(multi.reads, prm):
                assert row_bytes(rank_rows) == row_bytes(exp)
    finally:
        g.close()
