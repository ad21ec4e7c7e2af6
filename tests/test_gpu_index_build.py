"""The point cloud and the device index built on the GPU from the reference sequences
(smb_point_cloud_build / smb_point_cloud_build_part / smb_index_build) against the host build of
host_index.cc, which restates the reference's `sigmap -i`: the same points bit for bit, the same
parts for every rank, and the same mapped rows as an index built from the host cloud."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, Dataset, bits

pytestmark = pytest.mark.gpu


def crafted_reference(host):
    """Contigs too short for a window and just long enough; N runs and IUPAC codes (one in the
    first six bases); lowercase; a 300 bp element repeated until masked; a poly-A stretch and a
    short-period repeat over many tiles; stretches over {A,C} and {G,T} only; an all-masked contig."""
    rng = np.random.default_rng(11)

    def rand(n, alphabet=b"ACGT"):
        return bytes(np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), n)])

    element = rand(300)
    big = b"".join([
        b"ACGR" + rand(2000),
        b"N" * 50, rand(3000),
        b"ACRYKMSWBDHVN" * 3, rand(1500),
        rand(2000).lower(), rand(500),
        element * 40, rand(800),
        b"A" * 4000, rand(700),
        b"CAG" * 1500, rand(600),
        rand(6000, b"AC"), rand(400),
        rand(6000, b"GT"), rand(900),
        b"n" * 7, rand(1200).lower(), b"Y", rand(3000),
    ])
    seqs = [b"", rand(5), rand(6), rand(10), rand(11), rand(12), big, element * 3,
            rand(20000).lower(), b"N" + rand(9000)]
    return host.Reference([f"c{i}" for i in range(len(seqs))], seqs)


def flat_levels(model):
    """Pore-model levels with every 6-mer over {A,C} at one level and every one over {G,T} at
    another: the stretches over those alphabets then have equal z at every position (unmasked),
    so the selection keeps nothing there and tiles pass their state on without converging."""
    lv = np.array(model[0], np.float32, copy=True)
    h = np.arange(4096)
    digits = [(h >> (2 * k)) & 3 for k in range(6)]
    ac = np.all([(d == 0) | (d == 1) for d in digits], axis=0)
    gt = np.all([(d == 2) | (d == 3) for d in digits], axis=0)
    lv[ac] = lv[ac].mean(dtype=np.float64)
    lv[gt] = lv[gt].mean(dtype=np.float64)
    return lv


def big_levels(model):
    """Levels around 10^6 and one (AAAAAA) at 1.0: the smallest ulp of the table is 2^-23, so the
    sum of a strand's levels is an exact integer sum only for strands of a few hundred positions;
    the longer strands take the sequential sum."""
    lv = np.array(model[0], np.float32, copy=True) * np.float32(16384)
    lv[0] = 1.0
    return lv


@pytest.fixture(scope="module")
def dev():
    from sigmap_b200.mapper import Mapper
    m = Mapper(0)
    yield m
    m.close()


@pytest.fixture(scope="module")
def multi(host, model, tmp_path_factory):
    # the 7-contig genome of test_gpu_contig_shard.py
    return Dataset(host, model, tmp_path_factory.mktemp("multi_ib"),
                   [90000, 40000, 120000, 30000, 70000, 55000, 25000], 48, seed=21, noise=1.4,
                   min_bases=1500, max_bases=6000)


@pytest.fixture(scope="module")
def genomes(host, model, golden, multi):
    crafted = crafted_reference(host)
    return {
        "golden": (golden.genome(host), model[0]),
        "multi": (multi.ref, model[0]),
        "crafted": (crafted, model[0]),
        "crafted_flat": (crafted, flat_levels(model)),
        "crafted_big_levels": (crafted, big_levels(model)),
    }


def assert_same_cloud(got, exp):
    assert got[0].shape == exp[0].shape
    assert np.array_equal(got[0], exp[0])
    assert np.array_equal(bits(got[1]), bits(exp[1]))


@pytest.mark.parametrize("name", ["golden", "multi", "crafted", "crafted_flat", "crafted_big_levels"])
def test_cloud_equals_host(dev, host, genomes, name):
    ref, lv = genomes[name]
    dev.set_option("cloud_tile", 16384)
    exp = host.build_point_cloud(ref, lv)
    assert len(exp[0]) > 1000
    assert_same_cloud(dev.point_cloud(ref, lv), exp)
    st = dev.build_stats()
    assert st["points"] == len(exp[0]) and st["tile"] == 16384 and st["tiles"] > 0
    assert st["strands"] == 2 * sum(int(l) >= 11 for l in ref.lengths)
    if name == "crafted_big_levels":  # both ways of taking the mean ran
        assert 0 < st["strands_serial_mean"] < st["strands"]
    else:
        assert st["strands_serial_mean"] == 0


@pytest.mark.parametrize("tile", [32, 1000])
@pytest.mark.parametrize("name", ["golden", "crafted", "crafted_flat"])
def test_cloud_tiny_tiles(dev, host, genomes, name, tile):
    ref, lv = genomes[name]
    exp = host.build_point_cloud(ref, lv)
    dev.set_option("cloud_tile", tile)
    try:
        got = dev.point_cloud(ref, lv)
        st = dev.build_stats()
    finally:
        dev.set_option("cloud_tile", 16384)
    assert_same_cloud(got, exp)
    assert st["tile"] == tile and st["tiles"] >= 2 * sum(max(int(l) - 10, 0) for l in ref.lengths) // tile
    assert st["tiles_rewalked"] > 0  # the fix-up decided positions of the speculative walk anew
    if name != "golden":
        # the all-masked contig, the masked repeats, and (flat levels) the equal-z stretches
        # pass the state on over many consecutive tiles
        assert st["tiles_unconverged"] >= 6000 // tile


@pytest.mark.parametrize("world", [2, 3, 8])
def test_part_equals_host(dev, host, genomes, world):
    from sigmap_b200.shard import assign_contigs
    for name in ("multi", "crafted"):
        ref, lv = genomes[name]
        owner = assign_contigs(ref.lengths, world)
        for rank in range(world):
            exp_p = host.build_point_cloud_part(ref, lv, owner, rank)
            got_p = dev.point_cloud_part(ref, lv, owner, rank)
            try:
                exp, got = exp_p.arrays(), got_p.arrays()
            finally:
                exp_p.close()
                got_p.close()
            assert got["n_points_total"] == exp["n_points_total"], (name, rank)
            for k in ("pos", "own", "run_off", "run_first"):
                assert np.array_equal(got[k], exp[k]), (name, rank, k)
            assert np.array_equal(bits(got["val"]), bits(exp["val"])), (name, rank)


@pytest.fixture(scope="module")
def golden_pair(host, model, golden):
    """(index from the host cloud, index built on the device) over the golden genome."""
    from sigmap_b200.mapper import Mapper
    g = golden.genome(host)
    pos, val = host.build_point_cloud(g, model[0])
    a, b = Mapper(0), Mapper(0)
    a.set_index(pos, val)
    a.set_contigs(g.lengths)
    b.build_index(g, model[0])
    yield a, b
    a.close()
    b.close()


def row_bytes(rows):
    return [bytes(r) for r in rows]


def test_index_rows_equal_host_index(golden_pair, golden, host):
    from sigmap_b200.mapper import default_params, full_read_params
    a, b = golden_pair
    assert a.num_points == b.num_points
    reads = golden.reads(host)
    for prm in (default_params(), full_read_params()):
        exp = a.map_reads(reads, prm)
        assert sum(r.mapped for r in exp) > reads.n // 2
        assert row_bytes(b.map_reads(reads, prm)) == row_bytes(exp)
    assert b.build_stats()["ms_index"] > 0


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_build_rows_equal_unsharded(multi, model, world):
    from sigmap_b200 import shard
    from sigmap_b200.mapper import Mapper, default_params, full_read_params
    whole = Mapper(0)
    g = shard.ContigShardGroup([0] * world)
    try:
        whole.set_index(multi.pos, multi.val)
        whole.set_contigs(multi.ref.lengths)
        g.build_index(multi.ref, model[0])
        assert sorted(set(g.owner.tolist())) == list(range(world))
        for prm in (default_params(), full_read_params()):
            exp = whole.map_reads(multi.reads, prm)
            for rank_rows in g.map_reads(multi.reads, prm):
                assert row_bytes(rank_rows) == row_bytes(exp)
    finally:
        g.close()
        whole.close()


def test_more_ranks_than_contigs(host, model):
    """A rank that owns no contig keeps one padding leaf, as with the host-built part."""
    from sigmap_b200 import shard
    from sigmap_b200.mapper import default_params
    ref = host.sim_reference(5, [60000, 30000])
    reads = host.sim_reads(9, ref, 12, model=model)
    g = shard.ContigShardGroup([0, 0, 0])
    h = shard.ContigShardGroup([0, 0, 0])
    try:
        owner = [0, 1]
        g.build_index(ref, model[0], owner=owner)
        h.set_index_from_reference(ref, model[0], owner=owner)
        exp = h.map_reads(reads, default_params())
        got = g.map_reads(reads, default_params())
        for r in range(3):
            assert row_bytes(got[r]) == row_bytes(exp[r])
    finally:
        g.close()
        h.close()


def test_too_few_points_same_error_as_host(dev, host, model):
    from sigmap_b200.mapper import SigmapError
    ref = host.Reference(["tiny"], [b"ACGTTGCAACG"])  # one window per strand: 2 points
    pos, val = host.build_point_cloud(ref, model[0])
    assert np.array_equal(dev.point_cloud(ref, model[0])[0], pos)
    with pytest.raises(SigmapError) as e_host:
        dev.set_index(pos, val)
    with pytest.raises(SigmapError) as e_dev:
        dev.build_index(ref, model[0])
    code = lambda e: str(e.value).split("(")[1].split(")")[0]
    assert code(e_dev) == code(e_host)


def test_sharded_build_needs_a_group(dev, host, model):
    from sigmap_b200.mapper import SigmapError
    ref = host.sim_reference(3, [20000])
    with pytest.raises(SigmapError, match="shard group"):
        dev.build_index(ref, model[0], owner=[0])


def test_cli_index_on_gpu_is_byte_identical(host, golden, tmp_path):
    from sigmap_b200.host import MODEL_PATH
    exe = os.path.join(ROOT, "sigmap_b200", "bin", "sigmap")
    fasta = str(tmp_path / "ref.fa")
    golden.genome(host).write_fasta(fasta)
    outs = {}
    for tag, extra in (("host", []), ("gpu", ["--gpu", "0"])):
        prefix = str(tmp_path / tag)
        r = subprocess.run([exe, "-i", "-r", fasta, "-p", MODEL_PATH, "-o", prefix, *extra],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        outs[tag] = [open(prefix + ext, "rb").read() for ext in (".pt", ".si")]
    assert outs["gpu"][0] == outs["host"][0]
    assert outs["gpu"][1] == outs["host"][1]


@pytest.mark.parametrize("devices", [None, "0,0"])
def test_cli_map_index_from_ref(multi, tmp_path, devices):
    from sigmap_b200.host import MODEL_PATH
    exe = os.path.join(ROOT, "sigmap_b200", "bin", "sigmap")
    base = ["-m", "-r", multi.fasta, "-p", MODEL_PATH, "-s", multi.sigdir]
    extra = [] if devices is None else ["--gpus", devices, "--shard", "contigs"]
    exp, got = str(tmp_path / "x.paf"), str(tmp_path / "ref.paf")
    r = subprocess.run([exe, *base, "-x", multi.prefix, "-o", exp, *extra], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([exe, *base, "--index-from-ref", "-o", got, *extra], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    strip = lambda p: [[c for c in l.rstrip("\n").split("\t") if not c.startswith("mt:f:")]
                       for l in open(p)]
    rows = strip(exp)
    assert len(rows) == multi.reads.n
    assert strip(got) == rows
