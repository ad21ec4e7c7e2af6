"""The CUDA mapping path against the oracle on a repeat-rich reference (repeat_genome.py): dense
buckets (over two k_part_sort parts in a few thousand target positions), lookbacks cut by the
5 000-anchor band, link ranges deeper than what k_chain_prep stages, traceback into used anchors,
exactly tied chains on one contig, across contigs and across strands, and index points that are
bit-identical copies of each other.  test_oracle_repeats.py shows, without a GPU, that the oracle
meets every one of these on this data.  Bar: bit-exact chains, anchors, hit sets and PAF rows."""
import concurrent.futures
import os

import numpy as np
import pytest

import repeat_genome as RG
from conftest import bits, paf_cols, same_chains

pytestmark = pytest.mark.gpu

DIG, OFF, RNG = 8192.0, 10.0, 1437.976685


@pytest.fixture(scope="module")
def genome(host, model):
    return RG.RepeatGenome(host, model)


@pytest.fixture(scope="module")
def rmapper(genome):
    from sigmap_b200.mapper import Mapper
    m = Mapper(0)
    m.set_index(genome.pos, genome.val)
    m.set_contigs(genome.ref.lengths)
    yield m
    m.close()


@pytest.fixture(scope="module")
def oracle(port, genome):
    """the oracle's PAF rows, default and full-read rules"""
    return {"default": RG.oracle_rows(port, genome),
            "full": RG.oracle_rows(port, genome, RG.full_read_oracle_params(port))}


def test_multi_chunk_chains_on_repeats(rmapper, port, genome):
    """ChainBatch.GenerateChains against the oracle's GenerateChains, chunk after chunk with the
    chains carried over, every read sitting some rounds out (its chains must stay as they were)."""
    n_reads, n_chunks = genome.reads.n, 6
    feats = []
    for r in range(n_reads):
        pa = genome.pa(port, r)
        feats.append([port.generate_events(pa[c * 4000:(c + 1) * 4000])
                      for c in range(min(len(pa) // 4000, n_chunks))])

    def expected(r):  # the oracle's chains after each chunk of read r
        cl, off, out = port.new_chain_list(), 0, []
        for f in feats[r]:
            if len(f) > 50:
                out.append(port.generate_chains(genome.pos, genome.val, f, off, cl, n_targets=genome.ref.n))
                off += len(f)
            else:
                out.append(port.chains_py(cl))
        port.free_chain_list(cl)
        return out

    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        exp = list(ex.map(expected, range(n_reads)))
    batch = rmapper.ChainBatch(n_reads)
    done = [0] * n_reads
    rnd = checked = 0
    try:
        while any(done[r] < len(feats[r]) for r in range(n_reads)):
            slots = [r for r in range(n_reads) if done[r] < len(feats[r]) and (r + rnd) % 4]
            batch.GenerateChains(slots, [feats[r][done[r]] for r in slots])
            for r in range(n_reads):
                if r in slots:
                    assert same_chains(batch.chains(r), exp[r][done[r]]), f"read {r} chunk {done[r]}"
                    done[r] += 1
                    checked += 1
                elif done[r]:
                    assert same_chains(batch.chains(r), exp[r][done[r] - 1]), f"read {r} sat out round {rnd}"
            rnd += 1
    finally:
        batch.close()
    assert checked == sum(len(f) for f in feats) > 150


def test_rows_on_repeats_match_the_oracle(rmapper, genome, oracle):
    from sigmap_b200.mapper import default_params, full_read_params
    for mode, prm in (("default", default_params()), ("full", full_read_params())):
        rmapper.stats_reset()
        rows = rmapper.map_reads(genome.reads, prm)
        st = rmapper.stats()
        lines = rmapper.paf_lines(genome.reads, rows, genome.ref.names)
        for r in range(genome.reads.n):
            assert paf_cols(lines[r]) == paf_cols(oracle[mode][r]), f"{mode} read {r}"
        assert st["capped_queries"] == 0 and not any(row.flags & 1 for row in rows)


def test_dense_parts_take_the_part_sort_fallback_unforced(rmapper, genome, oracle):
    """A chunk over a tandem array overflows a k_part_sort part and one of its sub-ranges: the step's
    sort is redone by the generic kernels without any option set.  The per-entry k_seg_sort gives the
    same rows on these dense entries.  (Its own step-down, a coarse bin of over 10 240 anchors of one
    chunk, is not reached here: a chunk's anchors spread over the whole array, 11-15 kb.)"""
    def rows():
        rmapper.stats_reset()
        lines = rmapper.paf_lines(genome.reads, rmapper.map_reads(genome.reads), genome.ref.names)
        return [paf_cols(l) for l in lines], rmapper.stats()

    exp = [paf_cols(l) for l in oracle["default"]]
    got, st = rows()
    assert got == exp
    assert 0 < st["part_sort_steps"] < st["steps"], st
    rmapper.set_option("sort", "entry")
    try:
        got, st = rows()
    finally:
        rmapper.set_option("sort", "part")
    assert got == exp
    assert st["seg_sort_steps"] > 0, st


def test_search_finds_every_bit_identical_copy(rmapper, port, genome):
    """Windows of the two arrays and of B as queries: every window whose six values are bit-equal to
    the query (the other copies of the array unit; B's window in C and on D's - strand) is a hit at
    d2 = 0, and the hit sets (index + d2 bits) are the oracle's, with the lean kernel, the general
    kernel and a frontier limit that splits the queries between the two."""
    val = genome.val
    starts, a_pts = [], np.array(sorted(genome.points(0, 0)))
    for name in ("array0", "array1"):
        lo, hi = genome.spans[name]
        for at in np.linspace(lo + 400, hi - 400, 12).astype(int):
            starts.append(genome.window_index(0, 0, int(a_pts[np.searchsorted(a_pts, at)])))
    b_pts = sorted(p for p in genome.points(1, 0) if p >= 200)
    starts += [genome.window_index(1, 0, b_pts[k]) for k in np.linspace(0, len(b_pts) - 200, 8).astype(int)]
    q = np.stack([val[i:i + 6] for i in starts])
    windows = np.lib.stride_tricks.sliding_window_view(val.view(np.uint32), 6)
    copies = [np.flatnonzero((windows == q[k].view(np.uint32)).all(axis=1)) for k in range(len(q))]
    assert all(len(c) >= 100 for c in copies[:24]) and all(len(c) >= 3 for c in copies[24:])
    for radius in (0.08, 0.3):
        exp = [port.radius_search(val, x, radius=radius) for x in q]
        for name, value, reset in (("search", "lean", "lean"), ("search", "general", "lean"),
                                   ("front_cap", "72", "384")):
            rmapper.set_option(name, value)
            try:
                off, idx, d2 = rmapper.radiusSearch(q, radius=radius, cap=1 << 24)
            finally:
                rmapper.set_option(name, reset)
            for k, (ei, ed) in enumerate(exp):
                gi, gd = idx[off[k]:off[k + 1]], d2[off[k]:off[k + 1]]
                assert np.array_equal(gi, ei), f"{name}={value} r={radius} query {k}: hit set differs"
                assert np.array_equal(bits(gd), bits(ed)), f"{name}={value} r={radius} query {k}"
                at = np.searchsorted(gi, copies[k])
                assert np.array_equal(gi[at], copies[k]) and not gd[at].any(), f"query {k}: copies missed"


def test_read_until_rounds_on_repeats_match_offline(rmapper, genome):
    """Read-until on the repeat reads: raw samples in uneven slices, 16 channels; every decision
    equals the offline mapping of the same read."""
    n = 16
    offline = rmapper.map_reads(genome.reads)
    rmapper.stream_open(n)
    for ch in range(n):
        rmapper.stream_begin_read(ch, DIG, RNG, OFF)
    cursor, done = [0] * n, {}
    rngs = np.random.default_rng(5)
    for _ in range(200):
        chans, slices = [], []
        for ch in range(n):
            raw = genome.reads.read(ch)
            if ch in done or cursor[ch] >= len(raw):
                continue
            take = int(rngs.integers(1500, 6000))
            chans.append(ch)
            slices.append(raw[cursor[ch]:cursor[ch] + take])
            cursor[ch] += take
        if not chans:
            break
        dec, maps = rmapper.stream_round(chans, slices)
        for ch, d, m in zip(chans, dec, maps):
            if d:
                done[ch] = m
    rmapper.stream_close()
    assert done
    for ch, m in done.items():
        o = offline[ch]
        assert (m.mapped, m.contig, m.strand_plus, m.t_start, m.frag_len, m.chunks) == \
               (o.mapped, o.contig, o.strand_plus, o.t_start, o.frag_len, o.chunks), ch
