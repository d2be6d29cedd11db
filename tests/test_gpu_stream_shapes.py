"""Parity of the streamed path (MGATK_FLAG_ACCUMULATE parts + mgatk_stream_finish_device) with the oracle at the shapes the
one-batch suites pin and the streaming suites did not reach:

1. every streamed instance of the pileup kernels: compact, wide and indirect slots on contigs of 16 299, 16 577 (more
   chunks than the range table holds, sparse cells), 1 000 and 70 000 positions, with piles that pass 65 535 only in
   total on the last positions of the contig (above 65 535 at P = 70 000);
2. a slot layout that changes from part to part (compact, wide, indirect, compact), directly and through the BAM seam;
3. the carry planes at their limits: every cell deep, 64 deep cells (the default number of sets) and 65, a bulk cell
   whose units claim its set from many CTAs at once, a wrap inside the main kernel's accumulate epilogue, a coverage
   above 65 535 with no plane above it, and a Tn5 plane that wraps while no base plane does;
4. median depths on either side of every border k_median selects across (256, a shared or a different high byte, an
   unlisted 65 535, the overflow list), one batch and streamed.

Every part is cut on a start border, every output is filled with 0xA5 bytes before the stream begins, and each case
asserts on the oracle that it reaches the regime it is meant for.
"""
from __future__ import annotations

import numpy as np
import pytest

from mgatk2_b200.batch import ReadBatch
from mgatk2_b200.synth import make_whitelist, synth_batch
from tests.helpers import assert_result_equals_oracle
from tests.test_gpu_shapes import (assert_overflow_exact, engine, long_reads, make_params, pile, poison,  # noqa: F401
                                   run_both_entries, run_device_poisoned, to_lib_params)

pytestmark = pytest.mark.gpu


# ---------------------------------------------------------------------------------------------------------------- batches
def joined(batches):
    """Batches joined and stably sorted by start; their blobs are laid end to end and never repacked."""
    batches = [b for b in batches if b.n_records]
    shift, offs = 0, []
    for b in batches:
        offs.append(b.blob_off.astype(np.int64) + shift)
        shift += len(b.blob) // 16
    cat = {f: np.concatenate([getattr(b, f) for b in batches]) for f in ("pos", "tlen", "flag", "mapq", "bc_idx", "l_seq", "n_cigar")}
    order = np.argsort(cat["pos"], kind="stable")
    return ReadBatch(blob_off=np.concatenate(offs)[order].astype(np.uint32), blob=np.concatenate([b.blob for b in batches]),
                     **{f: v[order] for f, v in cat.items()})


def cut_at(batch, starts):
    """A start-sorted batch cut before each of `starts`: consecutive parts that share the batch's blob."""
    idx = [0, *np.searchsorted(batch.pos, starts, side="left").tolist(), batch.n_records]
    parts = [ReadBatch(pos=batch.pos[a:b], tlen=batch.tlen[a:b], flag=batch.flag[a:b], mapq=batch.mapq[a:b],
                       bc_idx=batch.bc_idx[a:b], l_seq=batch.l_seq[a:b], n_cigar=batch.n_cigar[a:b],
                       blob_off=batch.blob_off[a:b], blob=batch.blob) for a, b in zip(idx[:-1], idx[1:])]
    assert all(p.n_records for p in parts)
    for a, b in zip(parts[:-1], parts[1:]):
        assert a.pos[-1] < b.pos[0]
    return parts


def indirect_reads(rng, n, n_cells, lo, hi, L=2100):
    """n reads of L bases (indirect slots) with starts in [lo, hi), cells 0, 1, ... in turn."""
    b = long_reads(rng, n, np.arange(n_cells), L=L)
    b.pos = np.sort(rng.integers(lo, hi, n)).astype(np.int32)
    b.bc_idx = (np.arange(n) % n_cells).astype(np.int32)
    return b


def deep_tail(P, dist, cell=0):
    """Forward and reverse piles of one base in `cell`, 33 000 reads each at start P - 21 and again at P - 20: the A
    planes pass 65 535 on the last positions of the contig, but only once both starts are counted."""
    seq = "A" * (20 + 2 * dist)
    return [pile(33_000, P - 21, cell, seq, tlen0=1000), pile(33_000, P - 21, cell, seq, flag=16, tlen0=1000),
            pile(33_000, P - 20, cell, seq, tlen0=40_000), pile(33_000, P - 20, cell, seq, flag=16, tlen0=40_000)]


# ---------------------------------------------------------------------------------------------------------------- runs
def stream_poisoned(engine, parts, lp, overflow_capacity=1 << 16):
    """The parts through stream_begin / stream_add / stream_finish into 0xA5-filled outputs sized for the first part."""
    dout = engine.alloc_device_outputs(lp.n_cells, lp.mito_length, parts[0].n_records, overflow_capacity=overflow_capacity,
                                       max_read_extent=parts[0].max_read_extent())
    poison(dout)
    return engine.run_stream(parts, lp, dout), dout


def overflow_set(res):
    return {(int(c), int(pp), int(v)) for c, pp, v in zip(res.overflow["cell"], res.overflow["plane_pos"], res.overflow["value"])}


def assert_same_result(a, b):
    np.testing.assert_array_equal(a.planes, b.planes)
    np.testing.assert_array_equal(a.cell_qc, b.cell_qc)
    np.testing.assert_array_equal(a.base_totals, b.base_totals)
    assert a.stats == b.stats
    assert len(overflow_set(a)) == len(a.overflow) and overflow_set(a) == overflow_set(b)


def check_stream(engine, whole, parts, n_cells, one_batch=True, **kw):
    """The streamed parts against the oracle on the whole batch (dense, overflow list exact) and against one run_device
    of the whole batch. Returns (streamed result, its device outputs, params, oracle)."""
    from oracle.oracle import run_oracle
    assert sum(p.n_records for p in parts) == whole.n_records
    p = make_params(whole, n_cells, **kw)
    lp = to_lib_params(p)
    ora = run_oracle(whole, p, n_threads=8)
    res, dout = stream_poisoned(engine, parts, lp)
    assert_result_equals_oracle(res, ora)
    assert_overflow_exact(res, (ora.counts, ora.tn5, ora.coverage), np.arange(n_cells))
    if one_batch:
        one = engine.download(run_device_poisoned(engine, whole, lp), lp)
        assert_same_result(res, one)
    return res, dout, lp, ora


# ---------------------------------------------------------------------------------------------------------------- 1. instance matrix
MATRIX = {                                  # layout, P, parameters
    "atac50-16299": ("atac50", 16299, dict(min_distance_from_end=0)),
    "atac50-16577-gate": ("atac50", 16577, dict(min_distance_from_end=0, min_reads_per_cell=None)),
    "atac50-1000-raw": ("atac50", 1000, dict(min_distance_from_end=0, flags=1)),
    "atac50-70000": ("atac50", 70000, dict(min_distance_from_end=0)),
    "atac50-16569": ("atac50", 16569, dict(min_distance_from_end=0)),
    # position-only dedup keeps one read per start and strand, so those cases carry no deep piles
    "stress150-16299": ("stress150", 16299, dict(max_strand_bias=0.8, min_distance_from_end=10)),
    "stress150-16577": ("stress150", 16577, dict(max_strand_bias=0.8, min_distance_from_end=10, dedup_mode=1)),
    "stress150-1000": ("stress150", 1000, dict(max_strand_bias=0.8, min_distance_from_end=10, dedup_mode=1)),
    "stress150-70000": ("stress150", 70000, dict(max_strand_bias=0.8, min_distance_from_end=10)),
    "long-16299": ("long", 16299, dict()),
    "long-16577": ("long", 16577, dict()),
    "long-1000": ("long", 1000, dict()),
    "long-70000": ("long", 70000, dict()),
}


@pytest.mark.parametrize("case", list(MATRIX))
def test_streamed_instances(engine, case):
    """Four parts cut at P/3, 2P/3 and P - 20 (5P/6 without deep piles): 32 dense cells, 16 sparse ones (one unit across the whole contig), the
    deep piles of `deep_tail` in cell 0 split between the last two parts, and for the `long` layout about 40 reads of
    2 100 bases in the second part only. Against the oracle, one run_device, and the variant sums at 16 299 and 70 000."""
    from oracle.oracle import run_oracle
    layout, P, kw = MATRIX[case]
    kw = dict(kw, mito_length=P)
    seed = 7000 + P % 1013 + len(layout)
    profile = "stress150" if layout == "stress150" else "atac50"
    dense = synth_batch(32, 60_000, profile, seed=seed, mito_length=P)
    sparse = synth_batch(16, 400, profile, seed=seed + 1, mito_length=P)
    sparse.bc_idx = np.where(sparse.bc_idx >= 0, sparse.bc_idx + 32, sparse.bc_idx).astype(np.int32)
    pieces = [dense, sparse]
    deep = kw.get("dedup_mode", 0) != 1
    cuts = [P // 3, 2 * P // 3, P - 20 if deep else 5 * P // 6]
    if layout == "long":
        pieces.append(indirect_reads(np.random.default_rng(seed), 40, 32, cuts[0], cuts[1]))
    if deep:
        pieces += deep_tail(P, kw.get("min_distance_from_end", 5))
    whole = joined(pieces)
    parts = cut_at(whole, cuts)
    ext = [b.max_read_extent() for b in parts]
    if layout == "long":
        assert ext[1] >= 2100 and max(ext[0], ext[2], ext[3]) <= 56
    elif layout == "stress150":
        assert 56 < max(ext) <= 200
    else:
        assert max(ext) <= 56
    n_cells = 48
    if kw.get("min_reads_per_cell", 1) is None:             # a gate that some cells pass in total, never in one part
        n = run_oracle(whole, make_params(whole, n_cells, **{**kw, "min_reads_per_cell": 1}), n_threads=8, dense=False).cell_qc["n_reads"]
        gate = int(np.median(n[:32]))
        per_part = np.max([np.bincount(b.bc_idx[b.bc_idx >= 0], minlength=n_cells) for b in parts], axis=0)
        assert ((n >= gate) & (per_part < gate)).sum() >= 4 and ((n > 0) & (n < gate)).sum() >= 4
        kw["min_reads_per_cell"] = gate
    res, dout, lp, ora = check_stream(engine, whole, parts, n_cells, **kw)
    assert ora.cell_qc["n_reads"][32:].sum() > 0
    if deep:
        assert res.stats["n_overflow"] > 0
        assert (ora.counts[0, P - 10: P - 1, 0] > 65535).all()
    if P in (16299, 70000):
        from mgatk2_b200.variants import variant_sums
        from oracle.variants import oracle_variant_sums, reference_alleles
        from tests.test_gpu_variants import assert_sums_equal
        n = ora.cell_qc["n_reads"].astype(np.int64)
        alive = (n >= max(1, lp.min_reads_per_cell)) & (ora.cell_qc["sum_depth"] > 0)
        want = oracle_variant_sums(ora.counts, ora.coverage, reference_alleles(ora.base_totals), alive)
        assert_sums_equal(variant_sums((dout, lp), engine), want)


# ---------------------------------------------------------------------------------------------------------------- 2. layout changes between parts
@pytest.mark.parametrize("P", [16569, 16299])
def test_slot_layout_changes_between_parts(engine, P, tmp_path):
    """The same 24 cells in four parts whose slots are compact (50 bp), wide (150 bp with clips and indels), indirect
    (2 100 bp) and compact again: the workspace and the slot layout change from part to part, the planes carry over.
    Against the oracle and one run_device (wide slots throughout); then the same records as a BAM through the seam,
    streamed in parts of a sixth of the file, against the one-shot read of that file."""
    from mgatk2_b200 import BAMReader, PipelineConfig
    from mgatk2_b200.bamio import write_bam
    from tests.test_gpu_dropin import _same_cells
    n_cells = 24
    b1, b2, b3 = P // 4, P // 2, 3 * P // 4
    compact = synth_batch(n_cells, 40_000, "atac50", seed=P + 1, mito_length=P)
    compact = compact.take(np.nonzero((compact.pos < b1) | (compact.pos >= b3))[0])
    wide = synth_batch(n_cells, 20_000, "stress150", seed=P + 2, mito_length=P)
    wide = wide.take(np.nonzero((wide.pos >= b1) & (wide.pos < b2))[0])
    whole = joined([compact, wide, indirect_reads(np.random.default_rng(P), 48, n_cells, b2, b3)])
    parts = cut_at(whole, [b1, b2, b3])
    ext = [b.max_read_extent() for b in parts]
    assert ext[0] <= 56 and 56 < ext[1] <= 200 and ext[2] >= 2100 and ext[3] <= 56
    for b in parts:
        assert set(range(n_cells)) <= set(b.bc_idx[b.bc_idx >= 0].tolist())
    check_stream(engine, whole, parts, n_cells, mito_length=P, max_strand_bias=0.8)

    barcodes = make_whitelist(n_cells, seed=P)
    path = str(tmp_path / "possorted_bam.bam")
    write_bam(path, whole, barcodes, ref_lens=(248956422, P, 156040895))

    def read(**kw):
        reader = BAMReader(path, PipelineConfig(mito_length=P, max_strand_bias=0.8, sequential=True), set(barcodes),
                           barcode_list=barcodes, **kw)
        rbb, stats = reader.collect_reads_by_barcode()
        return reader, rbb, stats
    one, rbb_one, stats_one = read()
    streamed, rbb_parts, stats_parts = read(max_batch_records=whole.n_records // 6)
    assert not one.streamed and streamed.streamed
    assert stats_one == stats_parts
    _same_cells(rbb_one, rbb_parts)


# ---------------------------------------------------------------------------------------------------------------- 3. carry planes
def crossing_in_total(cells, s):
    """For each cell: 33 000 forward reads of A x 20 at start s and 33 000 at s + 1 (A forward reaches 66 000). Template
    lengths from 1 000 up: no duplicate of a background read (synth_batch's are at most 700)."""
    return [b for c in cells for b in (pile(33_000, s, int(c), "A" * 20, tlen0=1000), pile(33_000, s + 1, int(c), "A" * 20, tlen0=1000))]


def test_every_cell_deep(engine):
    """Three cells, three sets (the cap is the cell count): every cell claims one."""
    whole = joined(crossing_in_total(range(3), 4000))
    res, _, _, ora = check_stream(engine, whole, cut_at(whole, [4001]), 3, min_distance_from_end=0)
    assert (ora.counts[:, 4001:4020, 0, 0] == 66_000).all()


def test_sixty_four_deep_cells_and_sixty_five(engine):
    """70 cells, 64 sets: 64 cells that pass 65 535 only in total are exact; a 65th is refused (status 9), never silently
    saturated."""
    from mgatk2_b200.exceptions import PileupKernelError
    deep = np.random.default_rng(3).permutation(70)[:65]
    background = synth_batch(70, 20_000, "atac50", seed=64, mito_length=16569)
    whole = joined([background, *crossing_in_total(np.sort(deep[:64]), 8000)])
    res, _, _, ora = check_stream(engine, whole, cut_at(whole, [8001]), 70, one_batch=False, min_distance_from_end=0)
    assert len(np.unique(res.overflow["cell"])) == 64
    whole = joined([background, *crossing_in_total(deep, 8000)])
    lp = to_lib_params(make_params(whole, 70, min_distance_from_end=0))
    with pytest.raises(PileupKernelError) as e:
        stream_poisoned(engine, cut_at(whole, [8001]), lp)
    assert e.value.status == 9


@pytest.mark.parametrize("P", [16299, 16569])
def test_bulk_cell_claims_from_many_units(engine, P):
    """Cell 0: 3 600 forward reads of A x 20 at every start from 1 000 to 1 639, all in the second of four parts: that part
    alone takes the A forward plane to 72 000 at about 620 positions, so many k_pileup_big units of the cell claim its set
    at once. Cell 1 passes 65 535 inside the same part (70 000 reads at 1 300), cell 2 only in total (parts 3 and 4)."""
    background = synth_batch(8, 40_000, "atac50", seed=P, mito_length=P)
    bulk = [pile(3600, s, 0, "A" * 20, tlen0=1000) for s in range(1000, 1640)]
    whole = joined([background, *bulk, pile(70_000, 1300, 1, "A" * 20, tlen0=10_000), *crossing_in_total([2], 5000)])
    parts = cut_at(whole, [1000, 1640, 5001])
    assert parts[1].n_records > 2_300_000
    res, _, _, ora = check_stream(engine, whole, parts, 8, mito_length=P, min_distance_from_end=0)
    assert (ora.counts[0, :, 0, 0] >= 72_000).sum() >= 600
    assert set(np.unique(res.overflow["cell"]).tolist()) == {0, 1, 2}


def test_carry_claims_in_each_epilogue(engine):
    """Two parts cut at s0 + 10, three cells.
    Cell 0: 6 550 forward reads of A x 20 at each of s0 .. s0 + 9 (A forward 65 500 where they overlap, below the wrap),
    then 9 at each of s0 + 10 .. s0 + 19: 90 reads that fit a stage, so k_pileup_main's accumulate epilogue wraps.
    Cell 1: the same with ACGT x 5: coverage passes 65 535 at 7 positions while no counted plane passes 19 668, so the
    finish pass lists coverage entries and no set is needed.
    Cell 2: four groups (one base each) of 10 000 reverse 20 bp reads at s0 + 9 and 10 000 reverse 19 bp reads at s0 + 10,
    all ending at s0 + 28: Tn5 reverse reaches 80 000 there, split evenly between the parts; no base plane passes 20 000."""
    s0 = 6000
    pieces = []
    for c, seq in ((0, "A" * 20), (1, "ACGT" * 5)):
        pieces += [pile(6550, s, c, seq) for s in range(s0, s0 + 10)]
        pieces += [pile(9, s, c, seq) for s in range(s0 + 10, s0 + 20)]
    for g, base in enumerate("ACGT"):
        pieces += [pile(10_000, s0 + 9, 2, base * 20, flag=16, tlen0=1 + 10_000 * g),
                   pile(10_000, s0 + 10, 2, base * 19, flag=16, tlen0=1 + 10_000 * g)]
    whole = joined(pieces)
    parts = cut_at(whole, [s0 + 10])
    assert (parts[1].bc_idx == 0).sum() == 90
    res, _, _, ora = check_stream(engine, whole, parts, 3, min_distance_from_end=0)
    assert ora.counts[0, s0 + 19, 0, 0] == 65_590 and ora.counts[0, s0 + 9, 0, 0] == 65_500
    assert (ora.coverage[1] > 65535).sum() == 7 and ora.counts[1].max() <= 19_668 and ora.tn5[1].max() <= 65535
    assert ora.tn5[2, s0 + 28, 1] == 80_000 and ora.counts[2].max() == 20_000 and ora.coverage[2, s0 + 28] == 80_000


# ---------------------------------------------------------------------------------------------------------------- 4. medians
# per cell: depths of 20-position blocks, depths of single positions (1 bp reads), the (median_lo, median_hi) they give
MEDIANS = [
    ([255, 256], [], (255, 256)),                  # across the 256 border
    ([300, 400], [], (300, 400)),                  # same high byte: the second pass is reused
    ([511, 512], [], (511, 512)),                  # neighbouring high bytes
    ([1000, 65535], [], (1000, 65535)),            # a true 65 535, not in the overflow list
    ([65535, 65536], [], (65535, 65536)),          # across the saturation border
    ([65536, 131073], [], (65536, 131073)),        # both from the overflow list
    ([500, 700], [600], (600, 600)),               # 41 positions: one middle value, second pass
    ([], [300], (300, 300)),                       # n = 1
    ([], [300, 70000], (300, 70000)),              # n = 2
]


def test_bulk_depth_medians(engine):
    """Each cell of MEDIANS in one batch (host entry, and device entry with the base totals fused into k_median) and
    streamed in four parts that each hold one block or single position of every cell that has it (k_median without the
    fused totals)."""
    pieces = []
    for c, (blocks, singles, _) in enumerate(MEDIANS):
        pieces += [pile(d, 100 + 40 * j, c, "A" * 20) for j, d in enumerate(blocks)]
        pieces += [pile(d, 2000 + 10 * j, c, "A") for j, d in enumerate(singles)]
    whole = joined(pieces)
    n_cells = len(MEDIANS)
    host, dev, ora = run_both_entries(engine, whole, n_cells, min_distance_from_end=0)
    want = [m[2] for m in MEDIANS]
    assert list(zip(ora.cell_qc["median_lo"].tolist(), ora.cell_qc["median_hi"].tolist())) == want
    res, _, _, _ = check_stream(engine, whole, cut_at(whole, [140, 2000, 2010]), n_cells, min_distance_from_end=0)
    assert list(zip(res.cell_qc["median_lo"].tolist(), res.cell_qc["median_hi"].tolist())) == want
