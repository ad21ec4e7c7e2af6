"""A small reference rich in exact repeats, and reads that all lie on a repeat.

Every other dataset of the suite is uniform random sequence: the anchors of a chunk are spread
thin and every window has one true locus, so chains never tie.  This genome puts the chaining on
dense and tied input instead (buckets of over 10 000 anchors in a few thousand target positions,
lookbacks cut by the 5 000-anchor band, equal-score chains on one contig, across contigs and
across strands) while staying small enough for the brute-force oracle:

  A   220 kb random, holding
        two tandem arrays 2 kb apart (300 copies of a 50 bp unit, 300 of a 37 bp unit),
        a 6 kb segment and its copy 20 kb further on, same strand,
        a 4 kb segment and its reverse complement 30 kb further on;
  B   15 kb random;  C  a copy of B;  D  the reverse complement of B (its - strand is B);
  S   a 2 Mb satellite (12 000 copies of a 171 bp unit), masked whole: no point of the cloud;
  t5, t11, t12   contigs too short for a window (buckets that never hold an anchor).

The 11-mer mask drops k-mers more frequent than 0.0002 of all k-mers, and the hits of a query are
bounded by the copies of its 11-mer.  S counts its 2 M k-mers like a large genome would, which
puts the mask's limit near 460 copies: the arrays' 300 copies stay under it, while the oracle's
brute-force search still only scans the ~530 k points of A to D.  The repeats are kept out of B,
C and D (a triplicated array would reach the limit sooner).  `check_cloud` asserts on the point
cloud that the arrays survived the mask and that C and D carry B's points.

Reads are simulated from an excerpt of the genome (the arrays with their flanks, both copies of
each duplicated segment, and B), so every read lies on a repeat; a third of them at noise 0.3,
whose queries find most copies of their window, fill buckets past 10 000 anchors under the
default rules too.
"""
import concurrent.futures
import os

import numpy as np

SEED = 20261022
ARRAYS = ((50, 300), (37, 300))   # (unit length, copies)
SATELLITE = (171, 12000)          # (unit length, copies): contig S
FLANK = 1000
NOISE = (0.3, 1.0, 1.4)          # a third of the reads at each level


def _revcomp(s):
    return s[::-1].translate(bytes.maketrans(b"ACGT", b"TGCA"))


class RepeatGenome:
    def __init__(self, host, model, n_reads=36, min_bases=1500, max_bases=5000, seed=SEED):
        rng = np.random.default_rng(seed)

        def rand(n):
            return bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, n)])

        parts, self.spans = [], {}   # spans: name -> (start, end) on contig A

        def put(name, s):
            if name:
                at = sum(len(p) for p in parts)
                self.spans[name] = (at, at + len(s))
            parts.append(s)

        put(None, rand(40000))
        for k, (unit, copies) in enumerate(ARRAYS):
            put(f"array{k}", rand(unit) * copies)
            put(None, rand(2000))
        seg6 = rand(6000)
        put("seg6", seg6)
        put(None, rand(20000))
        put("seg6_copy", seg6)
        put(None, rand(30000))
        seg4 = rand(4000)
        put("seg4", seg4)
        put(None, rand(26000))
        put("seg4_rc", _revcomp(seg4))
        put(None, rand(220000 - sum(len(p) for p in parts)))
        a = b"".join(parts)
        b = rand(15000)
        sat = rand(SATELLITE[0]) * SATELLITE[1]
        names = ["A", "B", "C", "D", "S", "t5", "t11", "t12"]
        self.ref = host.Reference(names, [a, b, b, _revcomp(b), sat, rand(5), rand(11), rand(12)])
        self.pos, self.val = host.build_point_cloud(self.ref, model[0])
        check_cloud(self)

        # the excerpt the reads come from: every piece lies on a repeat
        lo, hi = self.spans["array0"][0] - FLANK, self.spans["array1"][1] + FLANK
        pieces = [a[lo:hi]] + [a[slice(*self.spans[n])] for n in ("seg6", "seg6_copy", "seg4", "seg4_rc")] + [b]
        excerpt = host.Reference([f"x{i}" for i in range(len(pieces))], pieces)
        per = [n_reads // len(NOISE) + (k < n_reads % len(NOISE)) for k in range(len(NOISE))]
        sets = [host.sim_reads(seed + 1 + k, excerpt, n, min_bases=min_bases, max_bases=max_bases,
                               noise=x, model=model)
                for k, (n, x) in enumerate(zip(per, NOISE))]
        raw = np.concatenate([s.raw for s in sets])
        off = np.cumsum([0] + [int(d) for s in sets for d in np.diff(s.read_off)], dtype=np.uint64)
        self.reads = host.ReadSet([f"rep_{i:03d}" for i in range(n_reads)], raw, off,
                                  host.DIGITISATION, host.RANGE, host.OFFSET)

    def pa(self, port, r):
        return port.raw_to_pa(self.reads.read(r), 8192.0, 10.0, 1437.976685)

    def points(self, contig, strand):
        """{position on the strand: z bits} of one (contig, strand)"""
        c = (self.pos >> np.uint64(33)).astype(np.int64)
        s = (self.pos & np.uint64(1)).astype(np.int64)
        p = ((self.pos >> np.uint64(1)) & np.uint64(0xFFFFFFFF)).astype(np.int64)
        k = (c == contig) & (s == strand)
        return dict(zip(p[k].tolist(), self.val[k].view(np.uint32).tolist()))

    def window_index(self, contig, strand, at):
        """index in the cloud of the window of (contig, strand) at position `at`"""
        key = (np.uint64(contig) << np.uint64(33)) | (np.uint64(at) << np.uint64(1)) | np.uint64(strand)
        k = np.flatnonzero(self.pos == key)
        assert len(k) == 1
        return int(k[0])


def check_cloud(g):
    """The repeats survived the 11-mer mask, and C and D carry B's points bit for bit once the
    window selection (whose state runs on from the previous strand) has converged."""
    plus_a = g.points(0, 0)
    for k, (unit, copies) in enumerate(ARRAYS):
        lo, hi = g.spans[f"array{k}"]
        kept = sum(lo <= p < hi for p in plus_a)
        assert kept > 0.8 * (hi - lo - 5), f"array{k}: {kept} points of {hi - lo} positions (masked?)"
    b_plus, b_minus = g.points(1, 0), g.points(1, 1)
    skip = 64
    for contig, strand, expect in ((2, 0, b_plus), (2, 1, b_minus), (3, 1, b_plus), (3, 0, b_minus)):
        got = g.points(contig, strand)
        tail = {p: v for p, v in got.items() if p >= skip}
        assert tail == {p: v for p, v in expect.items() if p >= skip}, (contig, strand)
        assert len(tail) > 0.8 * len(expect)


def oracle_rows(port, g, params=None, counters=False):
    """The oracle's PAF row of every read (and the counters, summed over the reads), computed
    over a thread pool: the oracle keeps no global state and ctypes releases the GIL."""
    from oracle.oracle import ChainCounters

    def one(r):
        ctr = ChainCounters()
        m = port.streaming_map(g.pos, g.val, g.ref.n, g.ref.lengths, g.pa(port, r), params, ctr)
        line = port.format_paf(m, g.reads.names[r], g.ref.names[m.contig], int(g.ref.lengths[m.contig]), 0.0)
        return line, m, ctr

    with concurrent.futures.ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        out = list(ex.map(one, range(g.reads.n)))
    total = ChainCounters()
    for _, _, c in out:
        total.add(c)
    lines = [l for l, _, _ in out]
    maps = [m for _, m, _ in out]
    return (lines, maps, total.as_dict()) if counters else lines


def full_read_oracle_params(port):
    """the oracle's parameters for full-read mode (mapper.full_read_params)"""
    p = port.default_params()
    p.max_num_chunks, p.stop_ratio, p.stop_mean_ratio, p.stop_min_anchors = 100000, 1e30, 1e30, 2000000000
    return p
