"""The repeat genome (repeat_genome.py) reaches the branches of the chaining that uniform random
references never do.  Runs without a GPU: the oracle's counters show, before any GPU run, that the
GPU tests of test_gpu_repeats.py put the CUDA chaining on the band limit of the lookback, on
position-only link ranges deeper than the 1 152 predecessors k_chain_prep stages, on traceback into
used anchors and on ties of the end-candidate and primary-chain orders."""
import pytest

import repeat_genome as RG


@pytest.fixture(scope="module")
def genome(host, model):
    return RG.RepeatGenome(host, model)


def test_repeat_reads_reach_the_dense_and_tied_branches(genome, port):
    total = {}
    for prm in (None, RG.full_read_oracle_params(port)):
        _, _, ctr = RG.oracle_rows(port, genome, prm, counters=True)
        for k, v in ctr.items():
            total[k] = max(total.get(k, 0), v) if k.startswith(("max_", "longest_")) else total.get(k, 0) + v
    for k in ("walks_band", "deep_link_ranges", "traceback_hit_used", "end_ties", "primary_ties"):
        assert total[k] > 0, (k, total)
    assert total["max_bucket_anchors"] > 2 * 5120, total   # over two k_part_sort parts
    assert total["longest_walk"] == 5000, total
    # below the 5 000-hit cap: the rows are the reference's, not its KD-tree traversal order's
    assert total["max_query_hits"] < 5000, total
