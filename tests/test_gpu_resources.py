"""Device memory comes back: a stage call that fails after it has allocated its buffers frees
them, and a context's whole life (index, mapping, a chain batch, a read-until stream, close)
returns what it took.  Free memory is read with torch.cuda.mem_get_info; other processes share
the GPU, so every comparison is a median over several readings."""
import statistics

import numpy as np
import pytest

from sigmap_b200.mapper import Mapper, SigmapError

pytestmark = pytest.mark.gpu

MiB = 1 << 20
DIG, OFF, RNG = 8192.0, 10.0, 1437.976685


def free_bytes():
    import torch
    return torch.cuda.mem_get_info(0)[0]


def test_failed_stage_call_frees_its_buffers(mapper, small):
    """smb_stage_radius sizes its hit buffers by `cap` (about 2 GB of keys and distances at
    cap = 2^26) and only then learns that the search found more hits than that.  Its error
    return must hand those buffers back."""
    rng = np.random.default_rng(11)
    starts = rng.integers(0, len(small.val) - 5, 16384)
    q = np.stack([small.val[starts + k] for k in range(6)], 1)

    # d^2 < 1.5 around points of the cloud: several thousand hits per query (the stage hook does
    # not cap queries), about 10^8 in all
    def failing_call():
        with pytest.raises(SigmapError, match="more hits than cap"):
            mapper.radiusSearch(q, radius=1.5, cap=1 << 26)

    failing_call()
    drops = []
    for _ in range(6):
        before = free_bytes()
        failing_call()
        drops.append(before - free_bytes())
    assert statistics.median(drops) < 256 * MiB, f"free memory drops per failed call: {drops}"


def test_context_life_returns_its_memory(small, port):
    """Create, use every kind of workspace, close: four times over, free memory must come back
    to where the first cycle left it."""
    feats = [port.generate_events(small.pa(port, r)[:4000]) for r in range(4)]
    raw = [small.reads.read(ch)[:12000] for ch in range(4)]

    def life():
        m = Mapper(0)
        try:
            m.set_index(small.pos, small.val)
            m.set_contigs(small.ref.lengths)
            m.map_reads(small.reads)
            batch = m.ChainBatch(len(feats))
            batch.GenerateChains(list(range(len(feats))), feats)
            batch.close()
            m.stream_open(len(raw))
            for ch in range(len(raw)):
                m.stream_begin_read(ch, DIG, RNG, OFF)
            m.stream_round(list(range(len(raw))), raw)
            m.stream_close()
        finally:
            m.close()
        return free_bytes()

    after = [life() for _ in range(4)]
    moved = [abs(after[0] - a) for a in after[1:]]
    assert statistics.median(moved) < 256 * MiB, f"free memory after each cycle: {after}"
