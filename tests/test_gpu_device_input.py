"""Mapping raw signal that already lives in device memory (smb_map_reads_device, Mapper.map_device):
the rows equal those of the host path (smb_map_reads) bit for bit whatever the layout of the
caller's tensor, the tensor is only read, the samples are not uploaded, the call is ordered after
the caller's stream, the context's uploaded read set is invalidated, bad input is refused, and
contig-sharded contexts map their own device copies like the unsharded mapper."""
import ctypes as C

import numpy as np
import pytest

from conftest import Dataset

pytestmark = pytest.mark.gpu

MODES = ("default", "full")


def _params(mode):
    from sigmap_b200.mapper import default_params, full_read_params
    return default_params() if mode == "default" else full_read_params()


def _fields(rows):
    """every field of every row; fp32 fields as their bits"""
    from sigmap_b200 import _ffi as F
    out = []
    for r in rows:
        row = []
        for name, typ in F.Mapping._fields_:
            v = getattr(r, name)
            row.append(int(np.float32(v).view(np.uint32)) if typ is C.c_float else int(v))
        out.append(tuple(row))
    return out


def _tables(reads):
    off = reads.read_off
    return off[:-1].copy(), np.diff(off).astype(np.uint32)


def _map(m, raw, start, length, reads, mode, **kw):
    return _fields(m.map_device(raw, start, length, reads.digitisation, reads.range, reads.offset,
                                _params(mode), **kw))


@pytest.fixture(scope="module")
def dev_raw(small):
    import torch
    return torch.from_numpy(small.reads.raw).to("cuda:0")


@pytest.fixture(scope="module")
def host_rows(mapper, small):
    return {mode: _fields(mapper.map_reads(small.reads, _params(mode))) for mode in MODES}


@pytest.mark.parametrize("mode", MODES)
def test_rows_equal_the_host_path(mapper, small, dev_raw, host_rows, mode):
    start, length = _tables(small.reads)
    assert sum(r[0] for r in host_rows[mode]) > small.reads.n // 2  # most reads map
    assert _map(mapper, dev_raw, start, length, small.reads, mode) == host_rows[mode]


@pytest.mark.parametrize("mode", MODES)
def test_layouts(mapper, small, host_rows, mode):
    import torch
    reads = small.reads
    start, length = _tables(reads)
    rng = np.random.default_rng(5)
    total = len(reads.raw)

    # the samples start at an odd element offset inside a larger tensor
    big = torch.from_numpy(rng.integers(-32768, 32767, total + 20, dtype=np.int16)).to("cuda:0")
    big[7:7 + total] = torch.from_numpy(reads.raw).to("cuda:0")
    assert _map(mapper, big, start + np.uint64(7), length, reads, mode) == host_rows[mode], "odd offset"

    # reads stored in reverse order with gaps of noise between them; tables in the original order
    gaps = 1 + np.arange(reads.n) % 7
    rev_start = np.zeros(reads.n, np.uint64)
    pos = 0
    for r in reversed(range(reads.n)):
        pos += int(gaps[r])
        rev_start[r] = pos
        pos += int(length[r])
    buf = rng.integers(-32768, 32767, pos + 3, dtype=np.int16)
    for r in range(reads.n):
        buf[int(rev_start[r]):int(rev_start[r]) + int(length[r])] = reads.read(r)
    got = _map(mapper, torch.from_numpy(buf).to("cuda:0"), rev_start, length, reads, mode)
    assert got == host_rows[mode], "reversed with gaps"

    # a padded [n, stride] batch (odd stride, noise in the padding)
    stride = int(length.max()) + 5
    pad = rng.integers(-32768, 32767, (reads.n, stride), dtype=np.int16)
    for r in range(reads.n):
        pad[r, :length[r]] = reads.read(r)
    rows = mapper.map_device_padded(torch.from_numpy(pad).to("cuda:0"), length, reads.digitisation,
                                    reads.range, reads.offset, _params(mode))
    assert _fields(rows) == host_rows[mode], "padded batch"


def test_empty_reads_and_empty_call(mapper, small, dev_raw):
    """read_len 0 gives the unmapped row a zero-length host read gets; zero reads give no rows"""
    import torch
    from sigmap_b200.host import ReadSet
    reads = small.reads
    start, length = _tables(reads)
    empty = [0, 5, reads.n - 1]
    length[empty] = 0
    keep = np.concatenate([reads.read(r) if length[r] else reads.raw[:0] for r in range(reads.n)])
    off = np.zeros(reads.n + 1, np.uint64)
    off[1:] = np.cumsum(length)
    host = ReadSet(reads.names, keep, off, 1.0, 1.0, 0.0)
    host.digitisation, host.range, host.offset = reads.digitisation, reads.range, reads.offset
    exp = _fields(mapper.map_reads(host, _params("default")))
    got = _map(mapper, dev_raw, start, length, reads, "default")
    assert got == exp
    assert all(got[r][0] == 0 for r in empty)
    none = mapper.map_device(torch.zeros(0, dtype=torch.int16, device="cuda:0"), [], [], [], [], [])
    assert len(none) == 0


def test_buffer_untouched_and_no_sample_upload(mapper, small, dev_raw):
    reads = small.reads
    start, length = _tables(reads)
    before = dev_raw.clone()
    mapper.stats_reset()
    mapper.map_reads(reads, _params("default"))
    host_st = mapper.stats()
    mapper.stats_reset()
    _map(mapper, dev_raw, start, length, reads, "default")
    st = mapper.stats()
    assert bool((dev_raw == before).all())
    assert st["h2d_bytes"] < 64 * reads.n + 4096, st["h2d_bytes"]
    assert host_st["h2d_bytes"] > 2 * len(reads.raw)  # the host path does upload the samples
    assert st["samples"] == host_st["samples"] > 0
    assert st["ms_filter"] > 0


def test_ordered_after_the_callers_stream(mapper, small, dev_raw, host_rows):
    """The tensor is filled on a side stream that is still busy when the call is made: the call
    must wait for the copy, not map the zeros that were there before it."""
    import torch
    start, length = _tables(small.reads)
    dst = torch.zeros_like(dev_raw)
    torch.cuda.synchronize(0)
    side = torch.cuda.Stream(device=0)
    with torch.cuda.stream(side):
        torch.cuda._sleep(200_000_000)  # keeps the side stream busy for ~0.1 s
        dst.copy_(dev_raw)  # cudaMemcpyAsync, device to device
    got = _map(mapper, dst, start, length, small.reads, "default", stream=side)
    assert got == host_rows["default"]


def test_uploaded_read_set(mapper, small, dev_raw, host_rows):
    from sigmap_b200 import shard
    from sigmap_b200.mapper import SigmapError
    reads = small.reads
    start, length = _tables(reads)
    mapper.upload_reads(reads)
    _map(mapper, dev_raw, start, length, reads, "default")
    # the device call replaced the read set: nothing uploaded is left to map
    with pytest.raises(SigmapError, match=r"smb_map_uploaded failed \(-6\): no uploaded reads"):
        mapper.map_uploaded(_params("default"))
    # a fresh upload is mapped again, and it is that set that is mapped
    half = shard.shard_reads(reads, 2, 1)
    mapper.upload_reads(half)
    assert _fields(mapper.map_uploaded(_params("default"))) == _fields(mapper.map_reads(half, _params("default")))
    # the host and the device path alternated on one context
    for _ in range(2):
        for mode in MODES:
            assert _fields(mapper.map_reads(reads, _params(mode))) == host_rows[mode]
            assert _map(mapper, dev_raw, start, length, reads, mode) == host_rows[mode]


def test_rejected_input(mapper, small, dev_raw, host_rows, monkeypatch):
    import torch
    from sigmap_b200 import _ffi as F
    from sigmap_b200.mapper import SigmapError
    reads = small.reads
    start, length = _tables(reads)
    out = (F.Mapping * reads.n)()
    prm = _params("default")

    def c_call(ptr):
        return F.lib.smb_map_reads_device(mapper._ctx, ptr, F.ptr(start, F.u64p), F.ptr(length, F.u32p),
                                          F.ptr(reads.digitisation, F.f32p), F.ptr(reads.range, F.f32p),
                                          F.ptr(reads.offset, F.f32p), reads.n, C.byref(prm), out, None)

    def last_error():
        return F.lib.smb_last_error(mapper._ctx).decode()

    assert c_call(reads.raw.ctypes.data) == -1  # SMB_ERR_ARG
    assert "pageable host memory" in last_error()
    pinned = torch.from_numpy(reads.raw).pin_memory()
    assert c_call(pinned.data_ptr()) == -1
    assert "pinned host memory" in last_error()
    if torch.cuda.device_count() > 1:
        other = dev_raw.to("cuda:1")
        assert c_call(other.data_ptr()) == -1
        assert "device 1" in last_error()
        with pytest.raises(SigmapError, match="cuda:1"):
            mapper.map_device(other, start, length, reads.digitisation, reads.range, reads.offset)

    # the Python checks refuse before the library is called
    def no_call(*a):
        raise AssertionError("smb_map_reads_device was called")

    with monkeypatch.context() as mp:
        mp.setattr(F.lib, "smb_map_reads_device", no_call)
        bad = [(dev_raw.to(torch.int32), "torch.int16"),
               (torch.stack([dev_raw, dev_raw], 1)[:, 0], "contiguous"),
               (torch.from_numpy(reads.raw), "cuda:0"),
               (reads.raw, "torch tensor")]
        for raw, msg in bad:
            with pytest.raises(SigmapError, match=msg):
                mapper.map_device(raw, start, length, reads.digitisation, reads.range, reads.offset)
        with pytest.raises(SigmapError, match="ends past"):
            mapper.map_device(dev_raw[:-1], start, length, reads.digitisation, reads.range, reads.offset)
        with pytest.raises(SigmapError, match="one entry per read"):
            mapper.map_device(dev_raw, start, length[:-1], reads.digitisation, reads.range, reads.offset)
    # the refused calls left the context usable
    assert _map(mapper, dev_raw, start, length, reads, "default") == host_rows["default"]


@pytest.fixture(scope="module")
def multi(host, model, tmp_path_factory):
    # the contig-shard tests' data set: 7 contigs of uneven length, noise 1.4
    return Dataset(host, model, tmp_path_factory.mktemp("multi"),
                   [90000, 40000, 120000, 30000, 70000, 55000, 25000], 48, seed=21, noise=1.4,
                   min_bases=1500, max_bases=6000)


def test_contig_sharded_ranks_map_their_own_device_copies(multi):
    import torch
    from sigmap_b200 import shard
    from sigmap_b200.mapper import Mapper
    reads = multi.reads
    start, length = _tables(reads)
    whole = Mapper(0)
    g = shard.ContigShardGroup([0, 0])
    try:
        whole.set_index(multi.pos, multi.val)
        whole.set_contigs(multi.ref.lengths)
        g.set_index(multi.pos, multi.val, multi.ref.lengths)
        copies = {id(m): torch.from_numpy(reads.raw).to("cuda:0") for m in g.mappers}
        for mode in MODES:
            exp = _fields(whole.map_reads(reads, _params(mode)))
            assert sum(r[0] for r in exp) > reads.n // 2
            got = g._each(lambda m: _map(m, copies[id(m)], start, length, reads, mode))
            for rank_rows in got:
                assert rank_rows == exp
        assert all(m.stats()["exchanges"] > 0 for m in g.mappers)
    finally:
        g.close()
        whole.close()
