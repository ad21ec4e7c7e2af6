"""GPU parity tests against the committed golden vectors (outputs of the unmodified reference,
tests/make_golden.py) -- these run on the GPU box without /root/reference -- and of the
`sigmap` CLI drop-in against the reference CLI."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits, paf_cols, same_chains

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gmapper(golden, host, model):
    from sigmap_b200.mapper import Mapper
    g = golden.genome(host)
    pos, val = host.build_point_cloud(g, model[0])
    m = Mapper(0)
    m.set_index(pos, val)
    m.set_contigs(g.lengths)
    yield m, g, pos, val
    m.close()


def test_raw_to_pa_golden(gmapper, golden, host):
    m = gmapper[0]
    got = m.raw_to_pa(golden["spiked_raw"], host.DIGITISATION, host.OFFSET, host.RANGE)
    assert np.array_equal(bits(got), bits(golden["pa_spiked"]))
    raw, dig, off, rng = golden.real_read(0)
    assert np.array_equal(bits(m.raw_to_pa(raw, dig, off, rng)), bits(golden["pa_real0"]))


def _golden_chunks(m, golden, host):
    reads = golden.reads(host)
    pas = {}
    out = []
    for kind, r, c in golden["chunk_src"]:
        key = (int(kind), int(r))
        if key not in pas:
            if kind == 0:
                pas[key] = m.raw_to_pa(reads.read(int(r)), host.DIGITISATION, host.OFFSET, host.RANGE)
            else:
                raw, dig, off, rng = golden.real_read(int(r))
                pas[key] = m.raw_to_pa(raw, dig, off, rng)
        out.append(pas[key][int(c) * 4000:(int(c) + 1) * 4000])
    return out


def test_events_golden_simulated_and_real_signal(gmapper, golden, host):
    m = gmapper[0]
    chunks = _golden_chunks(m, golden, host)
    got = m.GenerateEvents(np.stack(chunks))
    for ci, g in enumerate(got):
        e = golden.chunk_features(ci)
        assert g.shape == e.shape and np.array_equal(bits(g), bits(e)), f"chunk {ci}"
    for k, ci in enumerate(golden["detect_ids"]):
        d = m.detect_events(chunks[int(ci)])
        assert np.array_equal(bits(d["tstat1"]), bits(golden[f"det{k}_t1"]))
        assert np.array_equal(bits(d["tstat2"]), bits(golden[f"det{k}_t2"]))
        assert np.array_equal(d["peaks"].astype(np.uint64), golden[f"det{k}_peaks"])
        assert np.array_equal(bits(d["means"]), bits(golden[f"det{k}_means"]))


def test_radius_search_golden_kdtree_hits(gmapper, golden):
    m = gmapper[0]
    for name, radius in (("r008", 0.08), ("r030", 0.30)):
        off, idx, d2 = m.radiusSearch(golden["queries"], radius=radius)
        for k in range(len(golden["queries"])):
            gi, gd = idx[off[k]:off[k + 1]], d2[off[k]:off[k + 1]]
            ei, ed = golden.hits(name, k)
            keep = np.abs(gd - np.float32(radius)) > 1e-5       # north_star's boundary allowance
            ekeep = np.abs(ed - np.float32(radius)) > 1e-5
            assert np.array_equal(gi[keep], ei[ekeep]), f"{name} query {k}"
            assert np.array_equal(bits(gd[keep]), bits(ed[ekeep]))


def test_generate_chains_golden(gmapper, golden):
    m = gmapper[0]
    feats = {}
    for ci, (kind, r, c) in enumerate(golden["chunk_src"]):
        if kind == 0:
            feats[(int(r), int(c))] = golden.chunk_features(ci)
    n_reads = 1 + max(r for r, _ in feats)
    batch = m.ChainBatch(n_reads)
    states = list(golden.chain_states())
    by_round = {}
    for r, c, exp in states:
        by_round.setdefault(c, []).append((r, exp))
    checked = 0
    for c in sorted(by_round):
        # the reference skips chunks with <= 50 features; those are absent from the golden list
        slots = [r for r, _ in by_round[c]]
        batch.GenerateChains(slots, [feats[(r, c)] for r in slots])
        for r, exp in by_round[c]:
            assert same_chains(batch.chains(r), exp), f"read {r} chunk {c}"
            checked += 1
    assert checked == len(states) >= 25
    batch.close()


def test_paf_rows_golden_default_and_full(gmapper, golden, host):
    from sigmap_b200.mapper import default_params, full_read_params
    m, g = gmapper[0], gmapper[1]
    reads = golden.reads(host)
    for mode, prm in (("default", default_params()), ("full", full_read_params())):
        rows = m.map_reads(reads, prm)
        for name, line in zip(reads.names, m.paf_lines(reads, rows, g.names)):
            assert paf_cols(line) == golden.paf[mode][name], f"{mode} {name}"


def test_cli_dropin_matches_reference_cli(ref, small, golden, host, tmp_path):
    """`sigmap -i` writes the reference's .pt byte for byte; `sigmap -m` on the reference-built
    index prints the reference's PAF rows (all columns and tags except the wall-clock mt): on the
    golden genome and reads against the stored rows of the reference CLI, and, where oracle/_ref
    was built, on fresh inputs against the live reference."""
    import hashlib
    from sigmap_b200.host import MODEL_PATH
    exe = os.path.join(ROOT, "sigmap_b200", "bin", "sigmap")
    gdir = tmp_path / "golden"
    (gdir / "sig").mkdir(parents=True)
    fasta, gidx = str(gdir / "ref.fa"), str(gdir / "idx")
    golden.genome(host).write_fasta(fasta)
    golden.reads(host).write_blow5(str(gdir / "sig" / "reads.blow5"))
    r = subprocess.run([exe, "-i", "-r", fasta, "-p", MODEL_PATH, "-o", gidx], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    assert hashlib.sha256(open(gidx + ".pt", "rb").read()).hexdigest() == str(golden["pt_sha256"])
    full_read = ["--max-num-chunks", "100000", "--stop-mapping", "1e30", "--stop-mapping-mean", "1e30",
                 "--min-num-anchors", "2000000000"]
    for mode, extra in (("default", []), ("full", full_read)):
        out = str(gdir / f"{mode}.paf")
        r = subprocess.run([exe, "-m", "-r", fasta, "-p", MODEL_PATH, "-x", gidx, "-s", str(gdir / "sig"),
                            "-o", out, "-t", "2"] + extra, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr[-400:]
        assert {l.split("\t")[0]: paf_cols(l) for l in open(out)} == golden.paf[mode], mode
    ours_idx = str(tmp_path / "ours")
    r = subprocess.run([exe, "-i", "-r", small.fasta, "-p", MODEL_PATH, "-o", ours_idx],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    assert open(ours_idx + ".pt", "rb").read() == open(small.prefix + ".pt", "rb").read()
    out = str(tmp_path / "ours.paf")
    r = subprocess.run([exe, "-m", "-r", small.fasta, "-p", MODEL_PATH, "-x", ours_idx, "-s", small.sigdir,
                        "-o", out, "-t", "4", "--stop-mapping=1.4"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    assert "Finished mapping in" in r.stderr
    ours = {l.split("\t")[0]: paf_cols(l) for l in open(out)}
    assert len(ours) == small.reads.n
    if ref is None:  # the stored rows above are the comparison with the reference
        return
    rout = str(tmp_path / "ref.paf")
    rr = ref.cli(["-i", "-r", small.fasta, "-p", MODEL_PATH, "-o", str(tmp_path / "refidx")])
    assert rr.returncode == 0
    rr = ref.cli(["-m", "-r", small.fasta, "-p", MODEL_PATH, "-x", str(tmp_path / "refidx"), "-s", small.sigdir,
                  "-o", rout, "-t", "4"])
    assert rr.returncode == 0, rr.stderr[-400:]
    exp = {l.split("\t")[0]: paf_cols(l) for l in open(rout)}
    assert ours == exp
    # same row order too (by contig, then arrival; unmapped under contig 0 -- Q8), single-threaded
    rr = ref.cli(["-m", "-r", small.fasta, "-p", MODEL_PATH, "-x", str(tmp_path / "refidx"), "-s", small.sigdir,
                  "-o", rout, "-t", "1"])
    assert [l.split("\t")[0] for l in open(out)] == [l.split("\t")[0] for l in open(rout)]


@pytest.mark.parametrize("shard", ["reads", "contigs"])
def test_cli_multi_device_modes_match_single_device(small, tmp_path, shard):
    """`sigmap -m --gpus LIST --shard reads|contigs` (one context and host thread per entry; the
    list may repeat a device, which is how a one-GPU box tests it) prints the single-device PAF."""
    from sigmap_b200.host import MODEL_PATH
    exe = os.path.join(ROOT, "sigmap_b200", "bin", "sigmap")
    base = ["-m", "-r", small.fasta, "-p", MODEL_PATH, "-x", small.prefix, "-s", small.sigdir]
    one, many = str(tmp_path / "one.paf"), str(tmp_path / "many.paf")
    r = subprocess.run([exe, *base, "-o", one], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    r = subprocess.run([exe, *base, "-o", many, "--gpus", "0,0,0", "--shard", shard],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-400:]
    assert r.stderr.count("GPU 0:") == 3
    assert [paf_cols(l) for l in open(many)] == [paf_cols(l) for l in open(one)]
