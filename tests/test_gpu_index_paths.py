"""Every way of building the device index gives the same index, not just the same rows.  The C
ABI cannot read an index back, so two indexes are compared through what depends on their leaf and
node layout: the radius-search hits and their d2 bits over a fixed query set, and the counters of
one default mapping pass.  Each context sees the same calls in the same order, so the run-time
estimates the counters depend on agree too."""
import numpy as np
import pytest

from conftest import Dataset, bits

pytestmark = pytest.mark.gpu

LAYOUT_STATS = ("overflow_queries", "capped_queries", "hits", "anchors", "linked", "pending", "part_sort_steps")


@pytest.fixture(scope="module")
def multi(host, model, tmp_path_factory):
    # the 7-contig genome of test_gpu_contig_shard.py
    return Dataset(host, model, tmp_path_factory.mktemp("multi_ip"),
                   [90000, 40000, 120000, 30000, 70000, 55000, 25000], 48, seed=21, noise=1.4,
                   min_bases=1500, max_bases=6000)


@pytest.fixture(scope="module")
def queries(multi, port):
    qs = []
    for r in range(4):
        f = port.generate_events(multi.pa(port, r)[:4000])
        qs += [f[p:p + 6] for p in range(2, len(f) - 5, 2)]
    return np.stack(qs).astype(np.float32)


def search(m, q):
    off, idx, d2 = m.radiusSearch(q)
    return off, idx, bits(d2)


def layout_stats(m):
    st = m.stats()
    return {k: st[k] for k in LAYOUT_STATS}


def assert_same(got, exp, what):
    for a, b in zip(got[:3], exp[:3]):
        assert np.array_equal(a, b), what
    assert got[3] == exp[3], what


def test_host_cloud_index_equals_device_build(multi, model, queries):
    from sigmap_b200.mapper import Mapper, default_params
    a, b = Mapper(0), Mapper(0)
    try:
        a.set_index(multi.pos, multi.val)
        a.set_contigs(multi.ref.lengths)
        b.build_index(multi.ref, model[0])
        fp = []
        for m in (a, b):
            hits = search(m, queries)
            m.stats_reset()
            m.map_reads(multi.reads, default_params())
            fp.append(hits + (layout_stats(m),))
        assert len(fp[0][1]) > 1000 and fp[0][3]["anchors"] > 0
        assert_same(fp[1], fp[0], "smb_index_build against smb_index_set_points")
    finally:
        a.close()
        b.close()


@pytest.mark.parametrize("world", [2, 3])
def test_shard_paths_give_one_index_per_rank(multi, model, queries, world):
    from sigmap_b200 import shard
    from sigmap_b200.mapper import default_params
    groups = [shard.ContigShardGroup([0] * world) for _ in range(3)]
    try:
        whole, dev, part = groups
        whole.set_index(multi.pos, multi.val, multi.ref.lengths)
        dev.build_index(multi.ref, model[0], owner=whole.owner)
        part.set_index_from_reference(multi.ref, model[0], owner=whole.owner)
        fp = []
        for g in groups:
            hits = [search(m, queries) for m in g.mappers]
            for m in g.mappers:
                m.stats_reset()
            g.map_reads(multi.reads, default_params())
            fp.append([h + (layout_stats(m),) for h, m in zip(hits, g.mappers)])
        assert sum(len(h[1]) for h in fp[0]) > 1000
        for r in range(world):
            assert_same(fp[1][r], fp[0][r], f"rank {r}: smb_index_build(owner) against smb_index_set_points_sharded")
            assert_same(fp[2][r], fp[0][r], f"rank {r}: smb_index_set_points_part against smb_index_set_points_sharded")
    finally:
        for g in groups:
            g.close()


def test_cloud_in_falling_target_order(host, model, port):
    """A cloud whose points fall in target order inside every bucket (each bucket of a real cloud
    reversed): its bucket spans must still be 1 + the largest target, so the hit sets and the
    mapped rows are the oracle's over the same windows."""
    from sigmap_b200.mapper import Mapper
    ref = host.sim_reference(3, [120000, 60000])
    pos, val = host.build_point_cloud(ref, model[0])
    bucket = ((pos >> np.uint64(33)) << np.uint64(1)) | (pos & np.uint64(1))
    cut = np.flatnonzero(np.diff(bucket)) + 1
    order = np.concatenate([s[::-1] for s in np.split(np.arange(len(pos)), cut)])
    pos, val = np.ascontiguousarray(pos[order]), np.ascontiguousarray(val[order])
    assert (np.diff((pos >> np.uint64(1)).astype(np.int64)) < 0).sum() > len(pos) // 2
    reads = host.sim_reads(5, ref, 12, model=model)
    m = Mapper(0)
    try:
        m.set_index(pos, val)
        m.set_contigs(ref.lengths)
        q = []
        for r in range(2):
            f = port.generate_events(port.raw_to_pa(reads.read(r), 8192.0, 10.0, 1437.976685)[:4000])
            q += [f[p:p + 6] for p in range(2, len(f) - 5, 2)]
        q = np.stack(q)[:160]
        off, idx, d2 = m.radiusSearch(q)
        assert off[-1] > 0
        for k, x in enumerate(q):
            ei, ed = port.radius_search(val, x)
            assert np.array_equal(idx[off[k]:off[k + 1]], ei), f"query {k}: hit set differs"
            assert np.array_equal(bits(d2[off[k]:off[k + 1]]), bits(ed))
        rows = m.map_reads(reads)
        lines = m.paf_lines(reads, rows, ref.names)
        strip = lambda l: [c for c in l.rstrip("\n").split("\t") if not c.startswith("mt:f:")]
        for r in range(reads.n):
            pa = port.raw_to_pa(reads.read(r), 8192.0, 10.0, 1437.976685)
            e = port.streaming_map(pos, val, ref.n, ref.lengths, pa)
            exp = port.format_paf(e, reads.names[r], ref.names[e.contig], int(ref.lengths[e.contig]), 0.0)
            assert strip(lines[r]) == strip(exp), f"read {r}"
        assert sum(r.mapped for r in rows) > 0
    finally:
        m.close()
