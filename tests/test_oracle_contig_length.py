"""The oracle at a contig length other than chrM's: hand-computed known answers at P = 100.

The reference-generated goldens all use 16 569, so the places where P enters the oracle are pinned here by reads placed
around its borders: clipping of aligned blocks to [0, P) (pileup.py:57-65), the Tn5 bounds (pileup.py:43-50) and the
breadth denominator (processors.py:38). Every expected count below is written out by hand, one read per cell.
"""
import numpy as np
import pytest

from mgatk2_b200.batch import ReadBatch
from mgatk2_b200.processors import cell_qc_row
from oracle.oracle import make_params, run_oracle

P = 100
BASES = "ACGT"

# (pos, flag, seq, cigar): one record per cell, cell = index in this list
READS = [
    (95, 0, "ACGTACGTAC", [(0, 10)]),            # 0: forward, straddles P: 95..99 kept, 100..104 clipped
    (99, 0, "GGGGG", [(0, 5)]),                  # 1: starts at P - 1: one base
    (90, 16, "CCCCCCCCCC", [(0, 10)]),           # 2: reverse, ends at P - 1: Tn5 site at P - 1
    (91, 16, "TTTTTTTTTT", [(0, 10)]),           # 3: reverse, Tn5 site at P (dropped), bases 91..99 kept
    (-3, 0, "ACGTACGT", [(0, 8)]),               # 4: starts left of 0: query bases 3..7 land on 0..4, Tn5 site dropped
    (97, 0, "GGTTT", [(0, 2), (2, 5), (0, 3)]),  # 5: deletion 99..103 across P, the block after it (104..106) is beyond P
    (98, 16, "AAAAAA", [(0, 6)]),                # 6: reverse, straddles P: 98, 99 kept, Tn5 site 103 dropped
    (100, 16, "CCCCC", [(0, 5)]),                # 7: reverse, starts at P: nothing counted, the cell has no coverage
]

# expected (position, base, strand) counts per cell with min_distance_from_end = 0, and Tn5 sites (position, strand)
EXP_BASES = {
    0: [(95, "A", 0), (96, "C", 0), (97, "G", 0), (98, "T", 0), (99, "A", 0)],
    1: [(99, "G", 0)],
    2: [(p, "C", 1) for p in range(90, 100)],
    3: [(p, "T", 1) for p in range(91, 100)],
    4: [(0, "T", 0), (1, "A", 0), (2, "C", 0), (3, "G", 0), (4, "T", 0)],
    5: [(97, "G", 0), (98, "G", 0)],
    6: [(98, "A", 1), (99, "A", 1)],
    7: [],
}
EXP_TN5 = {0: [(95, 0)], 1: [(99, 0)], 2: [(99, 1)], 3: [], 4: [], 5: [(97, 0)], 6: [], 7: []}

# min_distance_from_end = 2 (pileup.py:67-72): only query positions [2, L - 2) count
EXP_BASES_D2 = {
    0: [(97, "G", 0), (98, "T", 0), (99, "A", 0)],
    1: [],                                       # L = 5: query window [2, 3) holds q = 2, at position 101
    2: [(p, "C", 1) for p in range(92, 98)],
    3: [(p, "T", 1) for p in range(93, 99)],
    4: [(0, "T", 0), (1, "A", 0), (2, "C", 0)],  # q = 3, 4, 5 (q = 2 lies at -1)
    5: [],                                       # q = 2 is the first base after the deletion, beyond P
    6: [],                                       # q = 2, 3 lie at 100, 101
    7: [],
}


def _batch():
    recs = [dict(pos=pos, flag=flag, mapq=60, seq=seq, cigar=cig, tlen=0, bc_idx=c) for c, (pos, flag, seq, cig) in enumerate(READS)]
    recs.sort(key=lambda r: r["pos"])
    return ReadBatch.from_records(recs)


def _expected(exp_bases, exp_tn5):
    C = len(READS)
    counts = np.zeros((C, P, 4, 2), np.uint32)
    tn5 = np.zeros((C, P, 2), np.uint32)
    for c, lst in exp_bases.items():
        for p, b, s in lst:
            counts[c, p, BASES.index(b), s] += 1
    for c, lst in exp_tn5.items():
        for p, s in lst:
            tn5[c, p, s] += 1
    cov = counts.sum(axis=(2, 3))
    tn5[cov == 0] = 0                                    # pileup.py:152-153: a position without coverage is dropped with its Tn5 counts
    return counts, tn5, cov


@pytest.mark.parametrize("d,exp_bases", [(0, EXP_BASES), (2, EXP_BASES_D2)], ids=["d0", "d2"])
def test_oracle_known_answers_at_p100(d, exp_bases):
    batch = _batch()
    p = make_params(len(READS), min_distance_from_end=d, dedup_mode=2, mito_length=P, max_read_extent=batch.max_read_extent())
    ora = run_oracle(batch, p)
    counts, tn5, cov = _expected(exp_bases, EXP_TN5)
    np.testing.assert_array_equal(ora.counts, counts)
    np.testing.assert_array_equal(ora.tn5, tn5)
    np.testing.assert_array_equal(ora.coverage, cov)
    assert ora.stats["total_reads"] == ora.stats["filtered_reads"] == len(READS)
    np.testing.assert_array_equal(ora.cell_qc["n_reads"], np.ones(len(READS)))
    covered = (cov > 0).sum(axis=1)
    np.testing.assert_array_equal(ora.cell_qc["covered"], covered)
    np.testing.assert_array_equal(ora.cell_qc["sum_depth"], cov.sum(axis=1))
    np.testing.assert_array_equal(ora.cell_qc["max_depth"], cov.max(axis=1))
    np.testing.assert_array_equal(ora.base_totals, counts.sum(axis=(0, 3)).astype(np.int64))


def test_oracle_hand_values_at_p100():
    """A few entries spelled out, so that the tables above cannot drift together with a wrong helper."""
    batch = _batch()
    p = make_params(len(READS), min_distance_from_end=0, dedup_mode=2, mito_length=P, max_read_extent=batch.max_read_extent())
    ora = run_oracle(batch, p)
    assert ora.counts.shape == (8, 100, 4, 2)
    assert ora.coverage[0, 99] == 1 and ora.coverage[0].sum() == 5            # 95..99 of a 10-base read at 95
    assert ora.counts[1, 99, 2, 0] == 1 and ora.coverage[1].sum() == 1        # G at P - 1
    assert ora.tn5[2, 99, 1] == 1 and ora.tn5[2].sum() == 1                   # reverse site 90 + 10 - 1 = P - 1
    assert ora.tn5[3].sum() == 0 and ora.coverage[3].sum() == 9               # reverse site at P: dropped
    assert ora.counts[4, 0, 3, 0] == 1 and ora.coverage[4, :5].sum() == 5     # query base 3 (T) at position 0
    assert ora.coverage[5].sum() == 2 and ora.tn5[5, 97, 0] == 1              # deletion across P: two bases before it
    assert ora.coverage[6, 98] == 1 and ora.coverage[6, 99] == 1 and ora.tn5[6].sum() == 0
    assert ora.coverage[7].sum() == 0 and ora.cell_qc["sum_depth"][7] == 0 and ora.cell_qc["n_reads"][7] == 1
    # breadth = covered / P (processors.py:38)
    assert cell_qc_row("x", ora.cell_qc[3], P)["coverage_breadth"] == 9 / 100
    assert cell_qc_row("x", ora.cell_qc[0], P)["coverage_breadth"] == 0.05
