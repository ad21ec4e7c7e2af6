"""CPU tests (no GPU): the C-ABI library loads and exports every symbol include/sigmap_b200.h
declares, refuses to run without a CUDA device (no CPU fallback), and the host-only helpers
(file formats, PAF text, simulator) behave like the reference's I/O layer."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, bits

HEADER = os.path.join(ROOT, "include", "sigmap_b200.h")


def _declared():
    txt = open(HEADER).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(smbh?_[a-z0-9_]+)\s*\(", txt)))


def test_every_declared_symbol_is_exported_and_bound():
    from sigmap_b200 import _ffi
    names = _declared()
    assert len(names) >= 45
    assert _ffi.MISSING == []
    for n in names:
        assert hasattr(_ffi.lib, n), f"{n} declared in the header but not exported"
        assert n in _ffi.PROTOTYPES, f"{n} has no ctypes prototype"
    nm = subprocess.run(["nm", "-D", "--defined-only", _ffi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (smbh?_[a-z0-9_]+)", nm))
    assert set(names) <= exported
    # nothing of the test oracle is linked into the product
    assert "orc_" not in nm and "liboracle" not in subprocess.run(
        ["ldd", _ffi.LIB_PATH], capture_output=True, text=True).stdout


def test_struct_sizes_match_header(tmp_path):
    from sigmap_b200 import _ffi
    src = '#include "sigmap_b200.h"\n#include <stdio.h>\nint main(){printf("%zu %zu %zu %zu %zu\\n",' \
          'sizeof(smb_params),sizeof(smb_mapping),sizeof(smb_chain),sizeof(smb_anchor),sizeof(smb_stats));}'
    exe = str(tmp_path / "smb_sizes")
    subprocess.run(["gcc", "-x", "c", "-", "-I", os.path.join(ROOT, "include"), "-o", exe],
                   input=src, text=True, check=True)
    got = [int(x) for x in subprocess.run([exe], capture_output=True, text=True).stdout.split()]
    assert got == [C.sizeof(_ffi.Params), C.sizeof(_ffi.Mapping), C.sizeof(_ffi.Chain),
                   C.sizeof(_ffi.Anchor), C.sizeof(_ffi.Stats)]


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from sigmap_b200 import _ffi
    from sigmap_b200.mapper import Mapper, SigmapError
    assert _ffi.lib.smb_device_count() == 0
    with pytest.raises(SigmapError, match="no CUDA device"):
        Mapper(0)
    ctx = C.c_void_p()
    assert _ffi.lib.smb_create(C.byref(ctx), 0) == -4 and not ctx.value


def test_product_never_imports_the_oracle():
    for base, _, files in os.walk(os.path.join(ROOT, "sigmap_b200")):
        for f in files:
            if f.endswith((".py", ".cc", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(base, f), errors="ignore").read()
                assert "oracle" not in txt.lower() or f in ("NOTICE.md",), f"{f} mentions the oracle"


def test_default_params_are_the_cli_defaults():
    from sigmap_b200.mapper import default_params
    p = default_params()
    assert (p.step_size, p.max_num_chunks, p.min_num_anchors, p.min_num_anchors_output) == (2, 30, 10, 10)
    assert np.float32(p.search_radius) == np.float32(0.08)
    assert (p.stop_mapping, p.stop_mapping_mean) == (np.float32(1.4), 5.0)
    assert p.stop_mapping_output == np.float32(1.2) and p.stop_mapping_mean_output == 5.0


def test_pore_model_and_fasta_round_trip(host, model, tmp_path):
    mean, stdv = model
    assert mean.shape == (4096,) and 50 < mean.min() < mean.max() < 130
    # first row of the bundled R9.4 model: AAAAAA 86.486336
    assert abs(mean[0] - 86.486336) < 1e-4 and stdv.min() > 0
    g = host.sim_reference(3, [1234, 77, 5000])
    p = str(tmp_path / "x.fa")
    g.write_fasta(p)
    back = host.Reference.read_fasta(p)
    assert back.names == g.names and back.seqs == g.seqs
    assert set(b"".join(g.seqs)) <= set(b"ACGT")
    assert max(len(l) for l in open(p).read().split("\n")) <= 60  # 60-column FASTA


def test_blow5_round_trip_and_reference_reader(host, model, ref, tmp_path):
    g = host.sim_reference(4, [30000])
    reads = host.sim_reads(9, g, 5, min_bases=300, max_bases=900, model=model)
    assert reads.n == 5 and reads.read_off[-1] == len(reads.raw)
    d = tmp_path / "sig"
    d.mkdir()
    p = str(d / "r.blow5")
    reads.write_blow5(p)
    back = host.ReadSet.read_blow5(p)
    assert back.names == reads.names
    assert np.array_equal(back.raw, reads.raw) and np.array_equal(back.read_off, reads.read_off)
    assert np.array_equal(back.digitisation, reads.digitisation)
    assert np.array_equal(bits(back.range), bits(reads.range))
    # determinism: any slice of the read stream can be generated independently (rank sharding)
    part = host.sim_reads(9, g, 2, first_read=3, min_bases=300, max_bases=900, model=model)
    assert np.array_equal(part.read(0), reads.read(3)) and np.array_equal(part.read(1), reads.read(4))
    assert np.array_equal(part.truth, reads.truth[3:])


def test_blow5_version_and_signal_compression_are_checked(host, model, tmp_path):
    """Files of slow5 >= 0.2.0 carry a signal-compression byte (svb-zd by default in current
    slow5tools): anything this reader cannot decode is refused with a message that says why."""
    g = host.sim_reference(4, [30000])
    reads = host.sim_reads(13, g, 3, min_bases=300, max_bases=600, model=model)
    plain = str(tmp_path / "v010.blow5")
    reads.write_blow5(plain)
    data = bytearray(open(plain, "rb").read())
    assert tuple(data[6:9]) == (0, 1, 0)

    def variant(name, **patch):
        d = bytearray(data)
        for off, val in patch.items():
            d[int(off[1:])] = val
        path = str(tmp_path / name)
        open(path, "wb").write(d)
        return path

    # 0.2.0 with uncompressed signals: the read-group count moves by one byte, records are the same
    d020 = bytearray(data)
    d020[7] = 2
    d020[11:15] = d020[10:14]
    d020[10] = 0
    p020 = str(tmp_path / "v020.blow5")
    open(p020, "wb").write(d020)
    back = host.ReadSet.read_blow5(p020)
    assert back.names == reads.names and np.array_equal(back.raw, reads.raw)
    for path, words in ((variant("svb.blow5", b7=2, b10=1), "signal compression"),
                        (variant("v1.blow5", b6=1, b7=0), "unsupported BLOW5 version 1.0.0"),
                        (variant("zstd.blow5", b9=2), "record compression")):
        with pytest.raises(RuntimeError) as e:
            host.ReadSet.read_blow5(path)
        assert words in str(e.value), str(e.value)


def test_blow5_zlib_records_truncation_and_append(host, model, tmp_path):
    """zlib-compressed records (slow5lib's default) read like plain ones; a truncated file is an
    error, not a short read set; reading a second file appends."""
    import struct
    import zlib
    g = host.sim_reference(4, [30000])
    reads = host.sim_reads(11, g, 7, min_bases=300, max_bases=900, model=model)
    plain = str(tmp_path / "plain.blow5")
    reads.write_blow5(plain)
    data = open(plain, "rb").read()
    hdr_len = struct.unpack_from("<I", data, 64)[0]
    at, recs = 68 + hdr_len, []
    while data[at:at + 5] != b"5WOLB" or at + 5 != len(data):
        n = struct.unpack_from("<Q", data, at)[0]
        recs.append(data[at + 8:at + 8 + n])
        at += 8 + n
    assert len(recs) == reads.n
    head = bytearray(data[:68 + hdr_len])
    head[9] = 1  # record compression: zlib
    packed = str(tmp_path / "zlib.blow5")
    with open(packed, "wb") as f:
        f.write(head)
        for r in recs:
            c = zlib.compress(r)
            f.write(struct.pack("<Q", len(c)) + c)
        f.write(b"5WOLB")
    back = host.ReadSet.read_blow5(packed)
    assert back.names == reads.names and np.array_equal(back.raw, reads.raw)
    assert np.array_equal(back.read_off, reads.read_off)
    assert np.array_equal(bits(back.offset), bits(reads.offset))
    # truncated: no EOF marker / cut inside a record
    for cut in (len(data) - 5, len(data) - 400):
        bad = str(tmp_path / f"cut{cut}.blow5")
        open(bad, "wb").write(data[:cut])
        with pytest.raises(Exception):
            host.ReadSet.read_blow5(bad)
    # appending two files through the C ABI (what the CLI does for a signal directory)
    from sigmap_b200 import _ffi as F
    import ctypes as C
    r = F.Reads()
    assert F.lib.smbh_blow5_read(plain.encode(), C.byref(r)) == 0
    assert F.lib.smbh_blow5_read(packed.encode(), C.byref(r)) == 0
    try:
        assert r.n == 2 * reads.n
        off = np.ctypeslib.as_array(r.read_off, (r.n + 1,))
        raw = np.ctypeslib.as_array(r.raw, (int(off[-1]),))
        assert np.array_equal(raw, np.concatenate([reads.raw, reads.raw]))
        assert [r.names[i].decode() for i in range(r.n)] == reads.names * 2
    finally:
        F.lib.smbh_reads_free(C.byref(r))


def test_format_paf_rows(host):
    from sigmap_b200 import _ffi
    m = _ffi.Mapping(mapped=1, read_len=22979, q_start=58, q_end=432, strand_plus=1, contig=0,
                     t_start=49622, frag_len=369, mapq=60, chunks=1, n_chains=1, cm=20,
                     s1=77.451462, s2=0.0, sm=77.451462, ad=0.055596, at=18.4, aq=16.5)
    cols = host.format_paf(m, "read_00000", "contig_0", 60000, 1.5).rstrip("\n").split("\t")
    assert cols[:12] == ["read_00000", "22979", "58", "432", "+", "contig_0", "60000", "49622",
                         "49991", "22979", "369", "60"]
    assert cols[12].startswith("mt:f:") and cols[13:16] == ["ci:i:1", "sl:i:22979", "cm:i:20"]
    assert cols[16] == "nc:i:1" and cols[17] == "s1:f:77.451462"
    u = _ffi.Mapping(mapped=0, read_len=3999, mapq=61, chunks=1)
    cols = host.format_paf(u, "short", "", 0, 0.0).rstrip("\n").split("\t")
    assert cols[:12] == ["short", "3999"] + ["*"] * 9 + ["61"]
    assert [c[:5] for c in cols[12:]] == ["mt:f:", "ci:i:", "sl:i:"]


def test_point_cloud_parts_cover_the_whole_cloud(host, model):
    """smbh_build_point_cloud_part: every rank's part holds exactly the windows of its own contigs,
    with the values the whole cloud has there (including the windows that straddle into the next
    contig / strand, Q2), and the parts of all ranks together are every window once."""
    # short contigs too: one shorter than a window run, so trailing values cross several contigs
    genome = host.sim_reference(31, [40000, 25, 30000, 14, 12, 22000, 9000])
    level_mean = model[0]
    pos, val = host.build_point_cloud(genome, level_mean)
    n = len(pos)
    for world in (2, 3):
        from sigmap_b200 import shard
        owner = shard.assign_contigs(genome.lengths, world)
        seen = np.zeros(n - 5, np.int32)
        for rank in range(world):
            part = host.build_point_cloud_part(genome, level_mean, owner, rank)
            a = part.arrays()
            part.close()
            assert a["n_points_total"] == n
            ro = a["run_off"]
            for k in range(len(a["run_first"])):
                lo, hi, g0 = int(ro[k]), int(ro[k + 1]), int(a["run_first"][k])
                # a run is a verbatim stretch of the whole cloud
                assert np.array_equal(a["pos"][lo:hi], pos[g0:g0 + hi - lo])
                assert np.array_equal(a["val"][lo:hi].view(np.uint32), val[g0:g0 + hi - lo].view(np.uint32))
                own = a["own"][lo:hi].astype(bool)
                assert np.array_equal(own, owner[(a["pos"][lo:hi] >> np.uint64(33)).astype(np.int64)] == rank)
                # every own point that is a window of the whole cloud has its six values in the run
                idx = g0 + np.nonzero(own)[0]
                idx = idx[idx < n - 5]
                assert np.all(idx - g0 + 5 < hi - lo)
                seen[idx] += 1
        assert np.all(seen == 1)
