"""GPU tests of everything that ships but the default run never reaches, and of the hot path at
the scale of BASELINE.json's configs:

* every search / sort / DP path behind `smb_set_option` gives the rows the default path gives
  (which test_gpu_parity.py holds to the oracle bit for bit), and really ran;
* the 5 000-hit cap (spatial_index.cc:371-372, SURVEY.md H4): set sizes, flags, determinism;
* harder inputs (three contigs, noise 1.6, samples outside the pA window) against the oracle;
* PAF concordance with the UNMODIFIED reference binary on config 1 exactly as BASELINE.json
  writes it (2 Mbp, 1 000 reads, default flags, reference -t 4) and on a slice of config 3
  (12 Mbp x 16 contigs: the 7-level index).  Bar: north_star's >= 99.5 %; expected: identical.
"""
import os

import numpy as np
import pytest

from conftest import Dataset, bits, paf_cols

pytestmark = pytest.mark.gpu


def _lines(m, ds, params=None):
    return [paf_cols(l) for l in m.paf_lines(ds.reads, m.map_reads(ds.reads, params), ds.ref.names)]


PATHS = [
    # option, value, what must be visible in the stats of the run
    ("sort", "entry", lambda st: st["seg_sort_steps"] > 0 and st["part_sort_steps"] == 0),
    ("sort", "global", lambda st: st["seg_sort_steps"] == 0),
    ("runs_cap", "8", lambda st: st["part_sort_steps"] < st["steps"]),   # run tables overflow -> radix sort
    ("search", "general", lambda st: st["overflow_queries"] == st["queries"]),
    ("front_cap", "72", lambda st: 0 < st["overflow_queries"] < st["queries"]),
    ("sort_queries_min", "0", lambda st: True),    # Morton-ordered queries even on this small batch
    ("sort_queries_min", "4000000000", lambda st: True),  # ... and never
    ("dp_tiles", "0", lambda st: True),            # no per-tile DP pass (the large-batch configuration)
    ("dp_tiles", "100000000", lambda st: True),    # ... and always
    ("prep_rounds", "0", lambda st: st["pending"] == st["linked"] > 0),   # every linked anchor walked by k_chain_dp
    ("prep_rounds", "2", lambda st: 0 < st["pending"] < st["linked"]),
    ("prep_rounds", "5", lambda st: 0 < st["pending"] < st["linked"]),
    ("pipeline", "on", lambda st: True),           # wave-pipelined ticks (one wave on this small input)
    ("pipeline", "off", lambda st: True),
    ("dp_passes", "0", lambda st: True),   # the cooperative in-order DP path settles everything
    ("dp_passes", "3", lambda st: True),
    ("events", "thread", lambda st: True),
    ("events", "warp", lambda st: True),
    ("events_overlap", "0", lambda st: True),
]
RESET = {"pipeline": "auto", "prep_rounds": "1", "sort_queries_min": "200000", "dp_tiles": "4096", "sort": "part", "runs_cap": "0", "search": "lean", "front_cap": "384",
         "dp_passes": "1", "events": "auto", "events_overlap": "1"}


def test_every_shipped_path_gives_the_default_rows(mapper, small):
    from sigmap_b200.mapper import full_read_params
    base, linked = {}, {}
    for mode, prm in (("default", None), ("full", full_read_params())):
        mapper.stats_reset()
        base[mode] = _lines(mapper, small, prm)
        linked[mode] = mapper.stats()["linked"]
    for name, value, seen in PATHS:
        mapper.set_option(name, value)
        try:
            for mode, prm in (("default", None), ("full", full_read_params())):
                mapper.stats_reset()
                got = _lines(mapper, small, prm)
                st = mapper.stats()
                assert got == base[mode], f"{name}={value} ({mode}) changes PAF rows"
                assert seen(st), f"{name}={value} ({mode}): the path did not run: {st}"
                # the set of anchors with a gap-compatible predecessor does not depend on the path
                assert st["linked"] == linked[mode], f"{name}={value} ({mode}): linked anchors differ"
        finally:
            mapper.set_option(name, RESET[name])
    # unknown names, and the switches of paths that no longer ship, are rejected
    for name in ("no_such_option", "index", "stage", "prep_bound", "grab", "part_fill", "part", "dp"):
        with pytest.raises(Exception):
            mapper.set_option(name, "1")
    assert _lines(mapper, small) == base["default"]


def _device_input(reads):
    """a CUDA tensor of the reads' samples and the per-read tables Mapper.map_device takes"""
    import torch
    off = reads.read_off
    raw = torch.from_numpy(reads.raw).to("cuda:0")
    return raw, off[:-1].copy(), np.diff(off).astype(np.uint32)


def test_wave_pipelined_ticks_give_identical_rows(mapper, small):
    """Reads joining in waves (1 MB slices, seven reads per tick: survivors wait a tick and are carried
    forward as absent slots while the next wave's events run) give the rows of the one-batch run, with
    host buffers, with resident samples and with device input (filter-only slices over a CUDA tensor),
    default and full-read rules, with and without event overlap."""
    from sigmap_b200.mapper import full_read_params
    modes = (("default", None), ("full", full_read_params()))
    base = {mode: _lines(mapper, small, prm) for mode, prm in modes}
    names = small.ref.names
    reads = small.reads
    raw, start, length = _device_input(reads)
    try:
        mapper.set_option("upload_slice_mb", "1")
        mapper.set_limits(max_batch_chunks=7)
        for pipe, overlap in (("on", "1"), ("on", "0"), ("off", "1")):
            mapper.set_option("pipeline", pipe)
            mapper.set_option("events_overlap", overlap)
            for mode, prm in modes:
                mapper.stats_reset()
                assert _lines(mapper, small, prm) == base[mode], f"pipeline={pipe} overlap={overlap} {mode}: host buffers"
                if pipe == "on":
                    assert mapper.stats()["steps"] >= small.reads.n // 7
                mapper.upload_reads(small.reads)
                rows = mapper.map_uploaded(prm)
                got = [paf_cols(l) for l in mapper.paf_lines(small.reads, rows, names)]
                assert got == base[mode], f"pipeline={pipe} overlap={overlap} {mode}: resident samples"
                rows = mapper.map_device(raw, start, length, reads.digitisation, reads.range, reads.offset, prm)
                got = [paf_cols(l) for l in mapper.paf_lines(reads, rows, names)]
                assert got == base[mode], f"pipeline={pipe} overlap={overlap} {mode}: device input"
    finally:
        mapper.set_option("pipeline", "auto")
        mapper.set_option("events_overlap", "1")
        mapper.set_option("upload_slice_mb", "64")
        mapper.set_limits(max_batch_chunks=32768)
    assert _lines(mapper, small) == base["default"]


def test_failed_mapping_call_leaves_the_context_usable(mapper, small):
    """A call of each entry point that fails mid-call (an anchor limit that one chunk overflows), with
    and without wave-pipelined ticks, reports the error; the next call on the same context, with a
    working limit, returns the rows of the default run."""
    from sigmap_b200.mapper import Mapper, SigmapError
    base = _lines(mapper, small)
    reads, names = small.reads, small.ref.names
    raw, start, length = _device_input(reads)

    # a mapper of its own: a failed call inflates the context's anchor estimate, so the working
    # limit is a moderate one (the default would size buffers for that estimate).  1 MB slices and
    # seven reads per tick: calls in several slices, which may still be queued when a call fails.
    m = Mapper(0)

    def host():
        return m.map_reads(reads)

    def resident():
        m.upload_reads(reads)
        return m.map_uploaded()

    def device():
        return m.map_device(raw, start, length, reads.digitisation, reads.range, reads.offset)

    try:
        m.set_index(small.pos, small.val)
        m.set_contigs(small.ref.lengths)
        m.set_option("upload_slice_mb", "1")
        m.set_limits(max_batch_chunks=7)
        for pipe in ("on", "off"):
            m.set_option("pipeline", pipe)
            for name, call in (("host", host), ("resident", resident), ("device", device)):
                m.set_limits(max_batch_anchors=16)
                with pytest.raises(SigmapError, match="one chunk overflows max_batch_anchors"):
                    call()
                m.set_limits(max_batch_anchors=1 << 24)
                got = [paf_cols(l) for l in m.paf_lines(reads, call(), names)]
                assert got == base, f"pipeline={pipe} {name}: rows after a failed call"
    finally:
        m.close()


def test_radius_search_paths_agree_with_the_oracle(mapper, port, small):
    """Hit sets (index + d2 bits) of the lean kernel, of the general kernel, and of the two
    together (a frontier limit that sends a share of the queries to the general kernel), on the
    index of `small` and on indexes of 6, 9 and 13 points (1 to 8 windows: one leaf, which keeps
    the windows' own order)."""
    from sigmap_b200.mapper import Mapper
    rng = np.random.default_rng(21)
    qs = []
    for r in range(8):
        f = port.generate_events(small.pa(port, r)[:4000])
        for p in range(2, len(f) - 5, 2):
            qs.append(f[p:p + 6])
    q = np.stack(qs)
    q = q[rng.permutation(len(q))]

    def agree(m, val, q, radius):  # -> hits
        exp = [port.radius_search(val, x, radius=radius) for x in q]
        for name, value in (("search", "lean"), ("search", "general"), ("front_cap", "72"),
                            ("sort_queries_min", "0")):
            m.set_option(name, value)
            try:
                off, idx, d2 = m.radiusSearch(q, radius=radius, cap=1 << 24)
            finally:
                m.set_option(name, RESET[name])
            for k, (ei, ed) in enumerate(exp):
                gi, gd = idx[off[k]:off[k + 1]], d2[off[k]:off[k + 1]]
                assert np.array_equal(gi, ei), f"{name}={value} r={radius} query {k}: hit set differs"
                assert np.array_equal(bits(gd), bits(ed))
        return sum(len(e[0]) for e in exp)

    for radius in (0.08, 0.3):
        hits = agree(mapper, small.val, q[:160], radius)
    assert hits > 10000  # radius 0.3: dense enough to matter
    tiny = Mapper(0)
    try:
        for n in (6, 9, 13):
            val = small.val[:n]
            tiny.set_index(small.pos[:n], val)
            w = np.stack([val[i:i + 6] for i in range(n - 5)])  # every window finds itself at d2 = 0
            tq = np.concatenate([w, w + rng.normal(0.0, 0.1, w.shape).astype(np.float32)])
            for radius in (0.08, 0.3):
                assert agree(tiny, val, tq, radius) >= len(w)
    finally:
        tiny.close()


def test_hit_cap_5000(mapper, port, small):
    """spatial_index.cc:371-372 keeps the first 5 000 hits of a query in KD-tree traversal order
    (H4: not reproducible by another index).  What is checked: below the cap, queries with
    thousands of hits still give the oracle's chains bit for bit; a query over the cap contributes
    exactly 5 000 anchors and is counted, reads with such a query are flagged, and the result is
    deterministic."""
    from conftest import same_chains
    from sigmap_b200.mapper import default_params
    n_reads = 8
    feats = [port.generate_events(small.pa(port, r)[:4000]) for r in range(n_reads)]

    def counts(radius):
        out = []
        for f in feats:
            q = np.stack([f[p:p + 6] for p in range(2, 2 * ((len(f) - 6) // 2) + 1, 2)])
            off, _, _ = mapper.radiusSearch(q, radius=radius, cap=1 << 26)
            out.append(np.diff(off.astype(np.int64)))
        return out

    # radius 0.5: hundreds of hits per query (frontiers beyond the lean kernel's slots, the general
    # kernel's big-query path), nothing at the cap: the oracle's chains, bit for bit
    radius = 0.5
    hq = counts(radius)
    assert max(int(h.max()) for h in hq) < 5000 and sum(int(h.sum()) for h in hq) > 300000
    batch = mapper.ChainBatch(n_reads)
    mapper.stats_reset()
    batch.GenerateChains(list(range(n_reads)), feats, default_params(search_radius=radius))
    st = mapper.stats()
    assert st["capped_queries"] == 0 and st["hits"] == sum(int(h.sum()) for h in hq)
    assert st["overflow_queries"] > 0
    for r in range(n_reads):
        cl = port.new_chain_list()
        exp = port.generate_chains(small.pos, small.val, feats[r], 0, cl, radius=radius, n_targets=small.ref.n)
        assert same_chains(batch.chains(r), exp), f"read {r} differs from the oracle at radius {radius}"
        port.free_chain_list(cl)
    # radius 1.2: a good share of the queries is over the cap
    radius = 1.2
    hq = counts(radius)
    over = [int((h >= 5000).sum()) for h in hq]
    assert sum(over) > 20, "radius too small to reach the cap"
    prm = default_params(search_radius=radius)
    batch.reset()
    mapper.stats_reset()
    batch.GenerateChains(list(range(n_reads)), feats, prm)
    st = mapper.stats()
    assert st["capped_queries"] == sum(over)
    assert st["hits"] == sum(int(np.minimum(h, 5000).sum()) for h in hq)
    first = [batch.chains(r) for r in range(n_reads)]
    batch.reset()
    batch.GenerateChains(list(range(n_reads)), feats, prm)
    for r in range(n_reads):
        assert same_chains(batch.chains(r), first[r]), "capped result is not deterministic"
    batch.close()
    # whole path: flags bit 0 on exactly the reads that had a capped query in a consumed chunk
    sub = type(small.reads)(small.reads.names[:n_reads], small.reads.raw[:int(small.reads.read_off[n_reads])],
                            small.reads.read_off[:n_reads + 1], 8192.0, 1437.976685, 10.0)
    rows = mapper.map_reads(sub, default_params(search_radius=radius, max_num_chunks=1))
    for r in range(n_reads):
        assert bool(rows[r].flags & 1) == (over[r] > 0), f"read {r}: flag {rows[r].flags}, capped queries {over[r]}"


def test_noisy_multi_contig_spiked_reads(host, model, port, tmp_path):
    """Three contigs, noise 1.6, a third of the reads carrying samples outside the (30, 200) pA
    window (incl. the raw values either side of both thresholds); default and full-read rules."""
    from sigmap_b200.mapper import Mapper, default_params, full_read_params
    ds = Dataset(host, model, tmp_path, [150000, 80000, 120000], 36, seed=99, noise=1.6,
                 min_bases=1500, max_bases=7000)
    rng = np.random.default_rng(3)
    raw = ds.reads.raw.copy()
    edge = np.array([159, 160, 161, 162, 1128, 1129, 1130, 1131, -32768, 32767, 0], np.int16)
    for r in range(0, ds.reads.n, 3):
        a, b = int(ds.reads.read_off[r]), int(ds.reads.read_off[r + 1])
        where = a + rng.choice(b - a, size=(b - a) // 150, replace=False)
        raw[where] = rng.choice(edge, size=len(where))
    reads = host.ReadSet(ds.reads.names, raw, ds.reads.read_off, host.DIGITISATION, host.RANGE,
                         host.OFFSET, ds.reads.truth)
    full = port.default_params()
    full.max_num_chunks, full.stop_ratio, full.stop_mean_ratio, full.stop_min_anchors = 100000, 1e30, 1e30, 2000000000
    m = Mapper(0)
    try:
        m.set_index(ds.pos, ds.val)
        m.set_contigs(ds.ref.lengths)
        for mode, gp, op in (("default", default_params(), None), ("full", full_read_params(), full)):
            lines = m.paf_lines(reads, m.map_reads(reads, gp), ds.ref.names)
            for i, name in enumerate(reads.names):
                pa = port.raw_to_pa(reads.read(i), host.DIGITISATION, host.OFFSET, host.RANGE)
                e = port.streaming_map(ds.pos, ds.val, ds.ref.n, ds.ref.lengths, pa, op)
                exp = port.format_paf(e, name, ds.ref.names[e.contig], int(ds.ref.lengths[e.contig]), 0.0)
                assert paf_cols(lines[i]) == paf_cols(exp), f"{mode} {name}"
    finally:
        m.close()


def _reference_concordance(host, model, ref, tmp, contig_lengths, n_reads, seed, threads, first_read=0,
                           max_bases=9000):
    """Map the same simulated reads with the unmodified reference CLI (its own index build, its own
    BLOW5 reader) and with the CUDA path; -> (paf_eval.concordance dict, rows flagged H4)."""
    from sigmap_b200 import paf_eval
    from sigmap_b200.host import MODEL_PATH
    from sigmap_b200.mapper import Mapper
    tmp = str(tmp)
    genome = host.sim_reference(seed, contig_lengths)
    fasta = os.path.join(tmp, "ref.fa")
    genome.write_fasta(fasta)
    reads = host.sim_reads(seed + 1, genome, n_reads, first_read=first_read, max_bases=max_bases, model=model)
    sig = os.path.join(tmp, "sig")
    os.makedirs(sig, exist_ok=True)
    reads.write_blow5(os.path.join(sig, "reads.blow5"))
    prefix = os.path.join(tmp, "idx")
    r = ref.cli(["-i", "-r", fasta, "-p", MODEL_PATH, "-o", prefix])
    assert r.returncode == 0, r.stderr[-400:]
    out = os.path.join(tmp, "ref.paf")
    r = ref.cli(["-m", "-r", fasta, "-p", MODEL_PATH, "-x", prefix, "-s", sig, "-o", out, "-t", str(threads)])
    assert r.returncode == 0, r.stderr[-400:]
    m = Mapper(0)
    try:
        m.load_index(prefix)          # the reference's own .pt
        m.set_contigs(genome.lengths)
        rows = m.map_reads(reads)
        lines = m.paf_lines(reads, rows, genome.names)
        st = m.stats()
    finally:
        m.close()
    res = paf_eval.concordance(paf_eval.read_paf(out), paf_eval.read_paf(lines))
    exp = {l.split("\t")[0]: paf_cols(l) for l in open(out)}
    res["identical_paf_rows"] = sum(paf_cols(l) == exp[n] for n, l in zip(reads.names, lines))
    res["flagged_h4"] = [n for n, row in zip(reads.names, rows) if row.flags & 1]
    res["stats"] = st
    return res


def test_config1_concordance_with_reference(host, model, ref, tmp_path):
    """BASELINE.json configs[0] as written: 2 Mbp, 1 000 reads, default flags, reference -t 4."""
    if ref is None:
        pytest.skip("oracle/_ref not built")
    res = _reference_concordance(host, model, ref, tmp_path, [2_000_000], 1000, seed=20251017, threads=4)
    assert res["in_both"] == res["reads"] == 1000
    assert res["fraction"] >= 0.995, res["discordant"][:10]
    # no query reaches the cap on 2 Mbp: the rows are the reference's, character for character
    assert not res["flagged_h4"]
    assert res["identical_paf_rows"] == 1000


def test_config3_slice_concordance_with_reference(host, model, ref, tmp_path):
    """A 300-read slice of BASELINE.json configs[2]: 12 Mbp x 16 contigs -> 23.9 M points, seven
    node levels (the top ones in shared memory, the general search kernel's large stacks), ~226
    hits per query, 32 buckets per read."""
    if ref is None:
        pytest.skip("oracle/_ref not built")
    res = _reference_concordance(host, model, ref, tmp_path, [750_000] * 16, 300, seed=20251017,
                                 threads=os.cpu_count() or 4)
    assert res["in_both"] == res["reads"] == 300
    assert res["fraction"] >= 0.995, res["discordant"][:10]
    # rows may only differ where a query hit the 5 000 cap (H4: traversal order is the KD-tree's)
    assert res["identical_paf_rows"] >= 300 - len(res["flagged_h4"])
    assert res["stats"]["queries"] > 50000
