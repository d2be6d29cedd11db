"""Host checks of the deletion definitions (DESIGN §8 "Deletions"): hand-computed answers of oracle/deletions.py, the
pairing rule of mgatk2_b200/deletions.find_deletions on hand-built histograms, the HGVS <-> (l, r) conversion and the
round trip of both files. No GPU."""
import math

import numpy as np
import pytest

from mgatk2_b200.batch import ReadBatch
from mgatk2_b200.deletions import (CANDIDATES_DTYPE, DeletionScan, breakpoints, breakpoints_to_hgvs, deletion_heteroplasmy,
                                   deletion_name, find_deletions, hgvs_to_breakpoints, read_deletion_candidates,
                                   read_deletions, write_deletion_candidates, write_deletions)
from oracle import deletions as od

L_, R_ = 100, 300                       # m.102_300del
P = 1000
CLS = {"clip_left": 0, "clip_right": 1, "gap": 2, "wt": 3}


def rec(pos, cigar, bc=0, flag=0, mapq=60, tlen=0, seq=None):
    qlen = sum(n for op, n in cigar if op in (0, 1, 4, 7, 8))
    return {"pos": pos, "cigar": cigar, "bc_idx": bc, "flag": flag, "mapq": mapq, "tlen": tlen,
            "seq": seq if seq is not None else "A" * qlen}


def counts_of(recs, n_cells=8, dedup_mode=0, **kw):
    recs = sorted(recs, key=lambda r: r["pos"])
    return od.scan(ReadBatch.from_records(recs), n_cells, P, [(L_, R_)], dedup_mode=dedup_mode, **kw)


CASES = [   # (cigar, pos, class) — every read in its own cell
    ([(0, 40), (4, 10)], 61, "clip_left"),                  # a1 = l, trailing clip
    ([(4, 8), (0, 40)], 300, "clip_right"),                  # a0 = r, leading clip
    ([(0, 21), (2, 199), (0, 20)], 80, "gap"),               # D over exactly [l + 1, r)
    ([(0, 22), (2, 198), (0, 20)], 80, "wt"),                # D one off: its first block covers l and l + 1
    ([(0, 20), (2, 199), (0, 20)], 80, "wt"),                # D [100, 299): not the gap; its last block covers r - 1, r
    ([(0, 20), (2, 200), (0, 20)], 80, None),                # D [100, 300): neither the gap nor a block over a breakpoint
    ([(0, 40)], 61, None),                                   # ends exactly at l without a clip
    ([(0, 40)], 90, "wt"),                                   # covers l, l + 1
    ([(0, 40)], 280, "wt"),                                  # covers r - 1, r
    ([(0, 40), (4, 4)], 61, None),                           # clip shorter than min_clip
    ([(5, 4), (4, 6), (0, 40)], 300, "clip_right"),          # H + S leading
    ([(0, 40), (4, 7), (5, 5)], 61, "clip_left"),            # S + H trailing
    ([(4, 5), (1, 2), (0, 40)], 300, "clip_right"),          # an I before the first M: sl = 5 (the I is not a clip)
    ([(3, 199), (0, 30)], 101, "gap"),                       # N over exactly [l + 1, r), no block before it
    ([(0, 30), (3, 199), (0, 30)], 71, "gap"),               # an N op counts as a gap
    ([(4, 60)], 300, None),                                  # span 0: no part
]


@pytest.mark.parametrize("k", range(len(CASES)))
def test_read_class(k):
    cigar, pos, want = CASES[k]
    c = counts_of([rec(pos, cigar, bc=0)], n_cells=1)["counts"][0, :, 0]
    exp = np.zeros(4, np.uint32)
    if want:
        exp[CLS[want]] = 1
    assert c.tolist() == exp.tolist()


def test_clip_geometry_and_histograms():
    seq_lead = "CAGTT" + "GG" + "A" * 40                     # S5 I2 M40: leading clip = CAGTT
    seq_trail = "A" * 40 + "TGCAN" + "CC"                    # M40 S5 S2 (two trailing S ops) then H
    seq_hs = "TTTTTTG" + "A" * 40                            # H3 S7 M40
    recs = [rec(300, [(4, 5), (1, 2), (0, 40)], bc=0, seq=seq_lead),
            rec(61, [(0, 40), (4, 5), (4, 2), (5, 9)], bc=1, seq=seq_trail),
            rec(300, [(5, 3), (4, 7), (0, 40)], bc=2, seq=seq_hs),
            rec(500, [(4, 61), (0, 40)], bc=3, seq="C" * 101),      # clip longer than SEQ? no: 61 <= 101, counted
            rec(700, [(0, 10), (4, 70)], bc=4, seq="C" * 80)]       # sr = 70 <= 80
    g = od.geometry(recs[0])
    assert (g["sl"], g["sr"], g["a0"], g["a1"]) == (5, 0, 300, 339)
    g = od.geometry(recs[1])
    assert (g["sl"], g["sr"], g["a1"]) == (0, 7, 100)
    g = od.geometry(rec(10, [(4, 9), (0, 5)], seq="A" * 8 + "A" * 5))  # l_seq 13 >= 9: kept
    assert g["sl"] == 9
    g = od.geometry({"pos": 10, "cigar": [(4, 20), (0, 5)], "seq": "A" * 10})   # sl > l_seq counts as 0
    assert g["sl"] == 0
    o = od.scan(ReadBatch.from_records(sorted(recs, key=lambda r: r["pos"])), 8, P, [(L_, R_)], find=True)
    assert o["start_clip"][300] == 2 and o["end_clip"][100] == 1 and o["start_clip"][500] == 1 and o["end_clip"][709] == 1
    ss, es = o["start_seq"], o["end_seq"]
    # leading clips read outward from the junction: SEQ[sl - 1 - j]
    assert ss[300, 0].tolist() == [0, 0, 1, 1] and ss[300, 1].tolist() == [0, 0, 0, 2]    # T(j0 of CAGTT) + G(j0 of ..G)
    assert ss[300, 4].tolist() == [0, 1, 0, 1]               # C of CAGTT, T of TTTTTTG
    assert ss[300, 5:7].sum(axis=1).tolist() == [1, 1] and ss[300, 7:].sum() == 0
    # trailing: SEQ[l_seq - sr + j]; N is not counted
    assert es[100, :7].tolist() == [[0, 0, 0, 1], [0, 0, 1, 0], [0, 1, 0, 0], [1, 0, 0, 0], [0, 0, 0, 0],
                                    [0, 1, 0, 0], [0, 1, 0, 0]]
    assert ss[500].sum() == 16 and es[709].sum() == 16       # at most MGATK_DEL_KMER bases
    assert o["counts"][0, :, :5].sum(axis=0).tolist() == [1, 1, 1, 0, 0]


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_dedup_modes_and_stage1(mode):
    clip_r = [(4, 8), (0, 40)]
    recs = [
        rec(300, [(0, 40)], bc=1, tlen=150), rec(300, clip_r, bc=1, tlen=150),                  # non-relevant first copy
        rec(61, [(0, 40), (4, 10)], bc=2, tlen=150, mapq=5), rec(61, [(0, 40), (4, 10)], bc=2, tlen=150),   # low mapq
        rec(300, [(0, 40)], bc=3, tlen=150), rec(300, clip_r, bc=3, tlen=-200),                  # |tlen| differs
        rec(300, [(0, 40)], bc=4, tlen=150), rec(300, clip_r, bc=4, tlen=150, flag=16),          # strand differs
        rec(300, clip_r, bc=8), rec(300, clip_r, bc=-1), rec(300, clip_r, bc=5, flag=0x4),
        rec(300, clip_r, bc=5, flag=0x100), rec(300, clip_r, bc=5, flag=0x800),
        rec(300, clip_r, bc=6, mapq=29),
    ]
    o = counts_of(recs, n_cells=8, dedup_mode=mode, min_mapq=30)["counts"][0]
    want = np.zeros((4, 8), np.uint32)
    want[1, 1] = mode == 2
    want[0, 2] = mode == 2
    want[1, 3] = mode in (0, 2)
    want[1, 4] = 1
    assert o.tolist() == want.tolist()


def test_min_clip_keyword():
    recs = [rec(61, [(0, 40), (4, 3)]), rec(300, [(4, 5), (0, 40)], bc=1)]
    assert counts_of(recs, min_clip=3)["counts"][0, :2, :2].tolist() == [[1, 0], [0, 1]]
    assert counts_of(recs, min_clip=6)["counts"][0].sum() == 0


def test_hgvs_conversion():
    assert hgvs_to_breakpoints(8470, 13446) == (8468, 13446)
    assert breakpoints_to_hgvs(8468, 13446) == (8470, 13446)
    assert deletion_name(8468, 13446) == "m.8470_13446del"
    assert breakpoints([(8470, 13446), (102, 300)]).tolist() == [[8468, 13446], [100, 300]]
    assert breakpoints(None).shape == (0, 2)


# ---- pairing on hand-built histograms ----------------------------------------------------------------------------
PP = 400


def _scan(ref_len=PP):
    K = 16
    return DeletionScan(np.zeros((0, 2), np.int32), np.zeros((0, 4, 1), np.uint32), np.zeros(ref_len, np.uint64),
                        np.zeros(ref_len, np.uint64), np.zeros((ref_len, K, 4), np.uint64),
                        np.zeros((ref_len, K, 4), np.uint64), ref_len, 5)


def _put(hist_seq, p, bases, reads=6):
    for j, b in enumerate(bases):
        hist_seq[p, j, "ACGT".index(b)] += reads


def test_pairing_left_side_repeats_and_right_preference():
    ref = list("A" * PP)
    motif = "CGTTGCATGC"                                     # 10 bases
    for at in (200, 260, 320):
        ref[at: at + 10] = motif
    s = _scan()
    s.end_clip[50] = 6
    _put(s.end_seq, 50, motif)
    c = find_deletions(s, "".join(ref))                       # no right candidate: the smallest match
    assert [(x["l"], x["r"], x["support"]) for x in c] == [(50, 200, "left")]
    s.start_clip[260] = 5                                     # a right candidate at the second repeat wins
    c = find_deletions(s, "".join(ref), min_match=10)
    assert [(x["l"], x["r"], x["support"]) for x in c] == [(50, 260, "left")]
    c = find_deletions(s, "".join(ref), min_length=220)        # r - l - 1 >= 220: only the third copy
    assert [(x["l"], x["r"]) for x in c] == [(50, 320)]
    ref[205] = "N"                                            # an N never matches: the first copy is gone
    s.start_clip[260] = 0
    c = find_deletions(s, "".join(ref))
    assert [(x["l"], x["r"]) for x in c] == [(50, 260)]


def test_pairing_ties_min_match_and_both():
    ref = list("T" * PP)
    ref[300:312] = "ACGTACGTACGA"
    ref[40:52] = "GGCATTCAGCCA"                               # read backwards from l = 51: ACCGACTTACGG
    s = _scan()
    s.end_clip[51] = 7
    _put(s.end_seq, 51, "ACGTACGTACGA", reads=3)
    s.end_seq[51, 0, 2] += 3                                  # tie A / G at j = 0: A (first of ACGT) wins
    s.start_clip[300] = 9
    _put(s.start_seq, 300, "ACCGACTTACGG")
    c = find_deletions(s, "".join(ref))
    assert len(c) == 1 and (c[0]["l"], c[0]["r"], c[0]["support"]) == (51, 300, "both")
    assert c[0]["reads_left"] == 7 and c[0]["reads_right"] == 9
    assert c[0]["consensus_left"] == "ACGTACGTACGA" and c[0]["consensus_right"] == "ACCGACTTACGG"
    assert c[0]["deletion"] == "m.53_300del" and (c[0]["first"], c[0]["last"], c[0]["length"]) == (53, 300, 248)
    assert len(find_deletions(s, "".join(ref), min_match=13)) == 0     # consensus of 12 < min_match
    assert len(find_deletions(s, "".join(ref), min_reads=10)) == 0
    s.end_clip[51] = 4                                         # below min_reads: right support alone
    c = find_deletions(s, "".join(ref))
    assert [(x["l"], x["r"], x["support"]) for x in c] == [(51, 300, "right")]


def test_pairing_consensus_stops_at_first_empty_offset():
    s = _scan()
    s.end_clip[10] = 6
    _put(s.end_seq, 10, "ACGTACGTAC")
    s.end_seq[10, 11, 0] = 6                                   # offset 10 empty: offset 11 is not part of it
    ref = ["T"] * PP
    ref[200:210] = "ACGTACGTAC"
    c = find_deletions(s, "".join(ref))
    assert len(c) == 1 and c[0]["consensus_left"] == "ACGTACGTAC" and c[0]["r"] == 200


def test_heteroplasmy_and_files_round_trip(tmp_path):
    counts = np.zeros((2, 4, 3), np.uint32)
    counts[0, :, 0] = [1, 2, 3, 4]              # del 6, wt 4
    counts[0, :, 2] = [0, 0, 0, 0]              # NaN, not written
    counts[1, :, 1] = [0, 0, 0, 5]              # 0.0
    scan = DeletionScan(np.array([[100, 300], [8468, 13446]], np.int32), counts, None, None, None, None, P, 5)
    t = deletion_heteroplasmy(scan)
    assert len(t) == 6 and t["heteroplasmy"][0] == 0.6 and math.isnan(t["heteroplasmy"][2])
    t2 = deletion_heteroplasmy(scan, deletions=[(8470, 13446)], cells=np.array([False, True, True]))
    assert t2["deletion"].tolist() == ["m.8470_13446del"] * 2 and t2["heteroplasmy"][0] == 0.0
    write_deletions(t, ["AAA-1", "CCC-1", "GGG-1"], tmp_path / "deletions.tsv.gz")
    back = read_deletions(tmp_path / "deletions.tsv.gz")
    assert [(r["barcode"], r["deletion"], r["clip_left"], r["clip_right"], r["gap"], r["wt"], r["heteroplasmy"])
            for r in back] == [("AAA-1", "m.102_300del", 1, 2, 3, 4, 0.6), ("CCC-1", "m.8470_13446del", 0, 0, 0, 5, 0.0)]
    cands = np.zeros(2, CANDIDATES_DTYPE)
    cands[0] = (100, 300, "m.102_300del", 102, 300, 199, "both", 7, 9, "ACGT", "TTGA")
    cands[1] = (8468, 13446, "m.8470_13446del", 8470, 13446, 4977, "left", 12, 0, "ACGTACGTACGTACGT", "")
    write_deletion_candidates(cands, tmp_path / "deletion_candidates.tsv.gz")
    assert read_deletion_candidates(tmp_path / "deletion_candidates.tsv.gz").tolist() == cands.tolist()
