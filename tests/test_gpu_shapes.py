"""Parity of the CUDA path with the oracle at the shapes real runs reach and the other suites do not: many skewed barcode
columns (two-digit partition, compact and wide slots, background barcodes with a handful of reads, long empty runs, a hot
spot), the cell-count limit, contig lengths other than chrM's (generic plane pitch, non-fused base totals beyond 65 535
positions), streaming over many columns, unaligned batch arrays, any blob layout and the 16-bit strand-bias filter.

Every device output is filled with 0xA5 bytes before a run, so an entry the kernels leave unwritten cannot pass for a
zero. Large cases compare sampled columns densely (a column's planes depend only on its own records: dedup and the
pileup are per barcode, readers.py:118-150, processors.py:20-55) and everything else through per-cell sums on the device.
"""
import ctypes
import os

import numpy as np
import pytest

from mgatk2_b200.batch import ReadBatch
from mgatk2_b200.engine import CELL_QC_DTYPE, OVERFLOW_DTYPE, STATS_FIELDS, DeviceBatch, PileupResult
from mgatk2_b200.synth import synth_batch
from tests.helpers import assert_result_equals_oracle

pytestmark = pytest.mark.gpu

QC_FIELDS = ("n_reads", "n_paired", "sum_depth", "covered", "max_depth", "median_lo", "median_hi")
STAT_KEYS = ("total_reads", "stage1_reads", "filtered_reads", "dup_with_length", "dup_position_only", "n_empty_seq")
PROFILE_LEN = {"atac50": 50, "atac70": 70, "stress150": 150}


@pytest.fixture(scope="module")
def engine():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    from mgatk2_b200.engine import PileupEngine
    eng = PileupEngine(0)
    yield eng
    eng.close()


def make_params(batch, n_cells, **kw):
    from oracle.oracle import make_params as mk
    return mk(n_cells, max_read_extent=batch.max_read_extent(), **kw)


def to_lib_params(p):
    from mgatk2_b200._lib import ParamsC
    return ParamsC(*[getattr(p, f) for f, _ in p._fields_])


def digit_bits(n_cells):
    """Bits of the two partition digits for n_cells (api.cu make_layout)."""
    bits = 1
    while (1 << bits) < n_cells:
        bits += 1
    return (bits, 0) if bits <= 11 else ((bits + 1) // 2, bits - (bits + 1) // 2)


# ---------------------------------------------------------------------------------------------------------------- batches
def pile(n, pos, cell, seq, flag=0, tlen0=1):
    """n copies of one read (one prototype blob) at `pos` of `cell`, template lengths tlen0, tlen0 + 1, ..."""
    proto = ReadBatch.from_records([dict(pos=0, flag=0, mapq=60, seq=seq, cigar=[(0, len(seq))], tlen=0, bc_idx=0)])
    return ReadBatch(pos=np.full(n, pos, np.int32), tlen=np.arange(tlen0, tlen0 + n, dtype=np.int32),
                     flag=np.full(n, flag, np.uint16), mapq=np.full(n, 60, np.uint8), bc_idx=np.full(n, cell, np.int32),
                     l_seq=np.full(n, len(seq), np.uint16), n_cigar=np.ones(n, np.uint16), blob_off=np.zeros(n, np.uint32),
                     blob=proto.blob)


def sorted_concat(parts):
    """Batches joined and stably sorted by pos (blobs packed in record order)."""
    whole = ReadBatch.concat(parts)
    return whole.take(np.argsort(whole.pos, kind="stable"))


def skewed_batch(n_columns, n_real, n_records, profile, seed, mito_length=16569):
    """synth_batch's cells on a seeded random set of `n_columns` columns, about 3 % of the stage-1 records moved to
    background columns drawn Zipf-like (most get 1-10 reads; duplicate keys move together), empty columns at 0, at
    n_columns - 1 and in runs of more than 64, exact duplicates of the first read of 300 background columns, and one hot
    spot of 5 000 reads of one column at one start with distinct template lengths. Returns (batch, info)."""
    rng = np.random.default_rng(seed)
    base = synth_batch(n_real, n_records, profile, seed=seed, mito_length=mito_length)
    P = mito_length
    empty = {0, n_columns - 1}
    for _ in range(3):                                          # runs of 80 empty columns
        a = int(rng.integers(1, max(2, n_columns - 81)))
        empty.update(range(a, min(a + 80, n_columns - 1)))
    b0, _ = digit_bits(n_columns)
    forced = [c for c in (2 ** b0 - 1, 2 ** b0, 2 ** b0 + 1, 12287, 12288, 12289) if 0 < c < n_columns - 1]
    empty -= set(forced)
    free = np.setdiff1d(np.arange(n_columns), np.array(sorted(empty)))
    forced = np.array(forced[:n_real], np.int64)
    rest = rng.permutation(np.setdiff1d(free, forced))
    real_cols = np.concatenate([forced, rest[: n_real - len(forced)]])
    background = rest[n_real - len(forced):]
    hot_col = int(background[0])
    background = background[1:]
    bc = base.bc_idx.astype(np.int64)
    new_bc = np.where(bc >= 0, real_cols[np.maximum(bc, 0)], bc)
    # ~3 % of the stage-1 keys (cell, start, strand, |tlen|) go to background columns, Zipf-like weights
    alive = np.nonzero(bc >= 0)[0]
    key = (((bc[alive] * (P + 64) + base.pos[alive]) * 2 + ((base.flag[alive] >> 4) & 1)) << 20) + np.abs(base.tlen[alive])
    uk, inv = np.unique(key, return_inverse=True)
    moved_key = rng.random(len(uk)) < 0.03
    w = 1.0 / np.arange(1, len(background) + 1) ** 0.8
    col_of_key = background[np.minimum(np.searchsorted(np.cumsum(w) / w.sum(), rng.random(len(uk))), len(background) - 1)]
    m = moved_key[inv]
    new_bc[alive[m]] = col_of_key[inv[m]]
    moved = ReadBatch(pos=base.pos, tlen=base.tlen, flag=base.flag, mapq=base.mapq, bc_idx=new_bc.astype(np.int32),
                      l_seq=base.l_seq, n_cigar=base.n_cigar, blob_off=base.blob_off, blob=base.blob)
    # an exact copy of the first stage-1 read of some background columns: a duplicate of the column's first slot
    s1 = np.nonzero((new_bc >= 0) & ((moved.flag & 0x904) == 0) & np.isin(new_bc, background))[0]
    first_of = {}
    for i in s1[np.lexsort((s1, moved.pos[s1]))]:
        first_of.setdefault(int(new_bc[i]), int(i))
    cols_with = np.array(sorted(first_of))
    dup_cols = rng.choice(cols_with, size=min(300, len(cols_with)), replace=False) if len(cols_with) else cols_with
    copies = moved.take(np.array([first_of[int(c)] for c in dup_cols], np.int64))
    L = PROFILE_LEN[profile]
    hot_pos = int(rng.integers(P // 4, P // 2))
    hot = pile(5000, hot_pos, hot_col, "".join(rng.choice(list("ACGT"), size=L)), flag=99)
    batch = sorted_concat([moved, copies, hot])
    assert batch.is_sorted()
    return batch, dict(real_cols=np.sort(real_cols), background=background, empty=np.array(sorted(empty)), hot_col=hot_col,
                       dup_cols=dup_cols)


# ---------------------------------------------------------------------------------------------------------------- device runs
def poison(dout):
    """0xA5 in every byte of every output: an entry the kernels do not write shows up as 0xA5A5."""
    import torch
    for t in (dout.planes, dout.cell_qc, dout.stats, dout.base_totals, dout.overflow):
        t.view(-1).view(torch.uint8).fill_(0xA5)


def run_device_poisoned(engine, batch, lp, overflow_capacity=1 << 16, dbatch=None):
    import torch
    dout = engine.alloc_device_outputs(lp.n_cells, lp.mito_length, batch.n_records, overflow_capacity=overflow_capacity,
                                       max_read_extent=lp.max_read_extent)
    poison(dout)
    engine.run_device(dbatch if dbatch is not None else engine.upload(batch), lp, dout)
    torch.cuda.synchronize()
    return dout


def partial_result(engine, dout, lp, cols):
    """Stats, QC rows, totals and the overflow list of a device run, and the planes of `cols` only."""
    import torch
    stats_np = dout.stats.cpu().numpy().view(np.uint64)
    rc = engine.lib.mgatk_check_stats(stats_np.ctypes.data)
    assert rc == 0, engine.lib.mgatk_status_string(rc).decode()
    stats = {k: int(v) for k, v in zip(STATS_FIELDS, stats_np)}
    qc = dout.cell_qc.cpu().numpy().view(CELL_QC_DTYPE)[: lp.n_cells]
    ovf = dout.overflow.cpu().numpy().view(OVERFLOW_DTYPE)[: min(stats["n_overflow"], dout.overflow_capacity)]
    cols = np.asarray(sorted(set(int(c) for c in cols)), np.int64)
    planes = dout.planes.view(torch.int16)[torch.from_numpy(cols).to(dout.planes.device)].cpu().numpy().view(np.uint16)
    res = PileupResult(planes, qc, stats, dout.base_totals.cpu().numpy(), ovf, lp.mito_length, lp.min_reads_per_cell)
    res.columns = cols
    return res


def device_plane_sums(dout, P):
    """Per cell: sum over [0, P) of every plane (int64 [C, 11]) and whether the padding [P, ppad) holds anything."""
    import torch
    C = dout.n_cells
    chunk = max(1, (1 << 28) // (4 * dout.planes.shape[1] * dout.planes.shape[2]))     # 256 MB of int32 at a time
    sums, pad = [], []
    for c0 in range(0, C, chunk):
        x = dout.planes[c0: c0 + chunk].view(torch.int16).to(torch.int32) & 0xFFFF
        sums.append(x[:, :, :P].sum(dim=2, dtype=torch.int64).cpu())
        pad.append((x[:, :, P:] != 0).flatten(1).any(dim=1).cpu())
        del x
    return torch.cat(sums).numpy(), torch.cat(pad).numpy()


# ---------------------------------------------------------------------------------------------------------------- comparisons
def plane_rows(res, cols):
    """uint32 [k, 11, P] planes of columns `cols` (sorted), saturated entries patched from the overflow list."""
    cols = np.asarray(cols, np.int64)
    if res.columns is None:
        rows = res.planes[cols]
    else:
        idx = np.searchsorted(res.columns, cols)
        assert np.array_equal(res.columns[idx], cols)
        rows = res.planes[idx]
    out = rows[:, :, : res.mito_length].astype(np.uint32)
    o = res.overflow[np.isin(res.overflow["cell"], cols)]
    if len(o):
        r = np.searchsorted(cols, o["cell"])
        out[r, o["plane_pos"] >> 24, o["plane_pos"] & 0xFFFFFF] = o["value"]
    return out


def assert_columns_equal_oracle(res, batch, params, cols):
    """Dense planes and QC rows of columns `cols` against the oracle run on those columns' records alone."""
    from oracle.oracle import make_params as mk, run_oracle
    cols = np.asarray(sorted(set(int(c) for c in cols)), np.int64)
    sub = batch.take(np.nonzero(np.isin(batch.bc_idx, cols))[0])
    sub.bc_idx[:] = np.searchsorted(cols, sub.bc_idx)
    p = mk(len(cols), min_baseq=params.min_baseq, min_mapq=params.min_mapq, min_distance_from_end=params.min_distance_from_end,
           dedup_mode=params.dedup_mode, max_strand_bias=params.max_strand_bias, min_reads_per_cell=params.min_reads_per_cell,
           mito_length=params.mito_length, max_read_extent=params.max_read_extent, flags=params.flags)
    ora = run_oracle(sub, p, n_threads=8)
    got = plane_rows(res, cols)
    k, P = len(cols), params.mito_length
    np.testing.assert_array_equal(got[:, :8].transpose(0, 2, 1).reshape(k, P, 4, 2), ora.counts, err_msg="base planes")
    np.testing.assert_array_equal(got[:, 8:10].transpose(0, 2, 1), ora.tn5, err_msg="tn5 planes")
    np.testing.assert_array_equal(got[:, 10], ora.coverage, err_msg="coverage plane")
    for f in QC_FIELDS:
        np.testing.assert_array_equal(res.cell_qc[f][cols], ora.cell_qc[f], err_msg=f)
    return ora


def assert_overflow_exact(res, ora_counts_tn5_cov, cells):
    """The overflow list holds exactly one entry per (cell, plane, pos) of `cells` whose oracle value is above 65 535,
    with that value, nothing else and no duplicates; the matching plane entries are 65 535."""
    counts, tn5, cov = ora_counts_tn5_cov
    cells = np.asarray(cells, np.int64)
    exp = set()
    for r, c in enumerate(cells):
        planes = np.concatenate([counts[r].reshape(-1, 8).T, tn5[r].T, cov[r][None]])      # [11, P]
        for pl, p in zip(*np.nonzero(planes > 65535)):
            exp.add((int(c), int(pl), int(p), int(planes[pl, p])))
    o = res.overflow
    got = [(int(c), int(pp) >> 24, int(pp) & 0xFFFFFF, int(v)) for c, pp, v in zip(o["cell"], o["plane_pos"], o["value"])]
    assert len(got) == len(set(got)), "duplicate overflow entries"
    assert set(got) == exp
    assert res.stats["n_overflow"] == len(exp)
    for c, pl, p, _ in exp:
        row = c if res.columns is None else int(np.searchsorted(res.columns, c))
        assert res.planes[row, pl, p] == 65535


def assert_global_equal_oracle(res, ora):
    for k in STAT_KEYS:
        assert res.stats[k] == ora.stats[k], (k, res.stats[k], ora.stats[k])
    for f in QC_FIELDS:
        np.testing.assert_array_equal(res.cell_qc[f], ora.cell_qc[f], err_msg=f)
    np.testing.assert_array_equal(res.base_totals, ora.base_totals)


def assert_device_planes_consistent(dout, res, ora_qc, P):
    """Over every cell: base planes and coverage add up to the oracle's sum_depth, dead cells hold only zeros (over the
    poison), the padding beyond P is zero. Cells with overflow entries are compared through their patched rows."""
    sums, pad = device_plane_sums(dout, P)
    assert not pad.any(), f"padding beyond P written in cells {np.nonzero(pad)[0][:10]}"
    deep = np.unique(res.overflow["cell"]) if len(res.overflow) else np.zeros(0, np.int64)
    ok = ~np.isin(np.arange(len(sums)), deep)
    sd = ora_qc["sum_depth"].astype(np.int64)
    np.testing.assert_array_equal(sums[ok, 10], sd[ok], err_msg="coverage sums")
    np.testing.assert_array_equal(sums[ok, :8].sum(axis=1), sd[ok], err_msg="base plane sums")
    dead = sd == 0
    assert not sums[dead].any(), f"dead cells with non-zero planes: {np.nonzero(dead & sums.any(axis=1))[0][:10]}"


def sample_columns(n_columns, info, ora, seed, n_random=48):
    """Both ends, both sides of the digit border, the shared-memory cap of k_cell_counts, an empty, a one-read, the
    deepest and the hot-spot column, some duplicated background columns, and random ones."""
    rng = np.random.default_rng(seed)
    b0, b1 = digit_bits(n_columns)
    cols = {0, n_columns - 1}
    if b1:
        cols |= {2 ** b0 - 1, 2 ** b0, 2 ** b0 + 1}
    cols |= {c for c in (12287, 12288, 12289) if c < n_columns}
    n = ora.cell_qc["n_reads"]
    cols.add(int(info["empty"][len(info["empty"]) // 2]))
    one = np.nonzero(n == 1)[0]
    if len(one):
        cols.add(int(one[0]))
    cols.add(int(np.argmax(n)))
    cols.add(info["hot_col"])
    cols |= {int(c) for c in info["dup_cols"][:8]}
    cols |= {int(c) for c in rng.choice(n_columns, size=min(n_random, n_columns), replace=False)}
    return sorted(c for c in cols if 0 <= c < n_columns)


def check_skewed(engine, batch, info, n_columns, P, seed, **kw):
    from oracle.oracle import run_oracle
    p = make_params(batch, n_columns, mito_length=P, **kw)
    lp = to_lib_params(p)
    ora = run_oracle(batch, p, n_threads=16, dense=False)
    cols = sample_columns(n_columns, info, ora, seed)
    dout = run_device_poisoned(engine, batch, lp)
    res = partial_result(engine, dout, lp, cols)
    assert_global_equal_oracle(res, ora)
    assert_device_planes_consistent(dout, res, ora.cell_qc, P)
    assert_columns_equal_oracle(res, batch, p, cols)
    del dout
    return res, ora


# ---------------------------------------------------------------------------------------------------------------- 1. many skewed columns, compact slots
_CACHE = {}


def cached(key, make):
    if key not in _CACHE:
        _CACHE.clear()                                   # one batch at a time: bounded host memory
        _CACHE[key] = make()
    return _CACHE[key]


COMPACT = {
    "c2049": dict(n_columns=2049, n_real=600, n=400_000, P=16569),
    "c12289": dict(n_columns=12289, n_real=2500, n=600_000, P=16569),
    "c20000_p16299": dict(n_columns=20000, n_real=3000, n=600_000, P=16299),
}


@pytest.mark.parametrize("dedup_mode", [0, 1, 2])
@pytest.mark.parametrize("shape", list(COMPACT))
def test_many_skewed_columns_compact(engine, shape, dedup_mode):
    c = COMPACT[shape]
    seed = 4100 + c["n_columns"]
    batch, info = cached(("compact", shape), lambda: skewed_batch(c["n_columns"], c["n_real"], c["n"], "atac50", seed,
                                                                  mito_length=c["P"]))
    assert batch.max_read_extent() <= 56
    res, ora = check_skewed(engine, batch, info, c["n_columns"], c["P"], seed + dedup_mode, dedup_mode=dedup_mode)
    n = ora.cell_qc["n_reads"]
    assert ((n >= 1) & (n <= 10)).sum() > 100
    if dedup_mode != 2:                                  # (no counters without dedup, readers.py:118)
        assert res.stats["dup_with_length"] > 0


def test_many_columns_mostly_dead(engine):
    """min_reads_per_cell = 50: most background columns are dead and must come out all zero over the poison."""
    c = COMPACT["c12289"]
    seed = 4100 + c["n_columns"]
    batch, info = cached(("compact", "c12289"), lambda: skewed_batch(c["n_columns"], c["n_real"], c["n"], "atac50", seed))
    res, ora = check_skewed(engine, batch, info, c["n_columns"], c["P"], seed + 7, min_reads_per_cell=50)
    n = ora.cell_qc["n_reads"]
    assert ((n > 0) & (n < 50)).sum() > 1000


# ---------------------------------------------------------------------------------------------------------------- 2. many columns, wide slots
WIDE = {"w2049": dict(n_columns=2049, n_real=500, n=250_000), "w5000": dict(n_columns=5000, n_real=1200, n=300_000)}


def long_reads(rng, n, cols, L=2100, P=16569):
    recs = [dict(pos=int(rng.integers(0, P - 200)), flag=int(rng.choice([0, 16, 99, 147])), mapq=60,
                 seq="".join(rng.choice(list("ACGT"), size=L)), cigar=[(0, L)], tlen=int(rng.integers(-500, 500)),
                 bc_idx=int(rng.choice(cols))) for _ in range(n)]
    recs.sort(key=lambda r: r["pos"])
    return ReadBatch.from_records(recs)


@pytest.mark.parametrize("dedup_mode", [0, 1, 2])
@pytest.mark.parametrize("shape", list(WIDE))
def test_many_skewed_columns_wide(engine, shape, dedup_mode):
    c = WIDE[shape]
    seed = 5100 + c["n_columns"]
    batch, info = cached(("wide", shape), lambda: skewed_batch(c["n_columns"], c["n_real"], c["n"], "stress150", seed))
    assert 56 < batch.max_read_extent() <= 200
    res, ora = check_skewed(engine, batch, info, c["n_columns"], 16569, seed + dedup_mode, dedup_mode=dedup_mode,
                            max_strand_bias=0.8, min_distance_from_end=10)
    if dedup_mode != 2:
        assert res.stats["dup_with_length"] > 0


def test_many_skewed_columns_wide_with_long_reads(engine):
    """A few 2 100 bp reads (indirect slots) in 2 049 columns: they travel through both digit passes."""
    rng = np.random.default_rng(61)
    batch, info = skewed_batch(2049, 400, 150_000, "stress150", 5200)
    batch = sorted_concat([batch, long_reads(rng, 60, rng.choice(info["real_cols"], size=40, replace=False))])
    assert batch.max_read_extent() >= 2100
    extra_cols = np.unique(batch.bc_idx[batch.l_seq == 2100])
    info["dup_cols"] = np.concatenate([extra_cols[:20], info["dup_cols"]])
    check_skewed(engine, batch, info, 2049, 16569, 5201, max_strand_bias=0.8, min_distance_from_end=10, dedup_mode=1)


# ---------------------------------------------------------------------------------------------------------------- 3. the cell-count limit
def test_cell_count_limit(engine):
    """2^21 + 1 columns (two 11-bit digits) on a 64-position contig; 2^22 + 1 are refused."""
    n_columns, P = (1 << 21) + 1, 64
    assert engine.lib.mgatk_workspace_bytes(1000, (1 << 22) + 1, 50) == -1
    assert engine.lib.mgatk_workspace_bytes(1000, n_columns, 50) > 0
    batch, info = skewed_batch(n_columns, 20_000, 300_000, "atac50", 77, mito_length=P)
    res, ora = check_skewed(engine, batch, info, n_columns, P, 78, dedup_mode=0)
    assert (res.cell_qc["n_reads"] > 0).sum() > 10_000


# ---------------------------------------------------------------------------------------------------------------- 4. contig lengths
def edge_piles(P):
    """A forward pile of 66 000 reads ending at P - 1 (cell 0), a reverse pile of 66 000 whose Tn5 site is P - 1
    (cell 1) and reverse reads whose site lies at P and beyond (cell 1)."""
    return [pile(66_000, P - 20, 0, "A" * 20), pile(66_000, P - 20, 1, "C" * 20, flag=16),
            pile(50, P - 19, 1, "G" * 20, flag=16, tlen0=100_000), pile(50, P - 10, 1, "T" * 20, flag=16, tlen0=200_000)]


def run_both_entries(engine, batch, n_cells, **kw):
    """Host entry and poisoned device entry: both dense against the oracle. Returns (host result, device result, oracle)."""
    from oracle.oracle import run_oracle
    p = make_params(batch, n_cells, **kw)
    lp = to_lib_params(p)
    ora = run_oracle(batch, p, n_threads=8)
    host = engine.run_host(batch, lp, overflow_capacity=1 << 16)
    assert_result_equals_oracle(host, ora)
    dout = run_device_poisoned(engine, batch, lp)
    dev = engine.download(dout, lp)
    assert_result_equals_oracle(dev, ora)
    assert not dev.planes[:, :, lp.mito_length:].any()
    return host, dev, ora


@pytest.mark.parametrize("profile", ["atac50", "stress150"])
@pytest.mark.parametrize("P", [16299, 16384, 16513, 1000, 70000])
def test_contig_lengths(engine, P, profile):
    n_cells = 48
    batch = synth_batch(n_cells, 60_000, profile, seed=900 + P % 97, mito_length=P)
    deep = P in (16299, 70000)
    if deep:
        batch = sorted_concat([batch, *edge_piles(P)])
    host, dev, ora = run_both_entries(engine, batch, n_cells, mito_length=P, min_distance_from_end=0 if deep else 5)
    assert ora.coverage.shape == (n_cells, P) and host.planes.shape[2] == (P + 63) // 64 * 64
    if deep:
        for res in (host, dev):
            assert_overflow_exact(res, (ora.counts, ora.tn5, ora.coverage), np.arange(n_cells))
        assert ora.tn5[1, P - 1, 1] >= 66_000 and ora.coverage[0, P - 1] >= 66_000
        assert ora.base_totals[P - 1, 0] >= 66_000


def test_chrm_without_fused_totals(engine):
    """The non-fused base-totals pass (k_base_totals + the overflow correction) at chrM length."""
    batch = sorted_concat([synth_batch(48, 60_000, "atac50", seed=911), *edge_piles(16569)])
    os.environ["MGATK_FUSED_TOTALS"] = "0"
    try:
        host, dev, ora = run_both_entries(engine, batch, 48, min_distance_from_end=0)
    finally:
        del os.environ["MGATK_FUSED_TOTALS"]
    assert_overflow_exact(dev, (ora.counts, ora.tn5, ora.coverage), np.arange(48))


# ---------------------------------------------------------------------------------------------------------------- 5. streaming with many columns
@pytest.mark.parametrize("profile", ["atac50", "stress150"])
def test_stream_many_columns(engine, profile):
    import torch
    from oracle.oracle import run_oracle
    n_columns = 2049
    batch, info = skewed_batch(n_columns, 400, 200_000, profile, 6100 + len(profile))
    kw = dict(max_strand_bias=0.8, min_distance_from_end=10) if profile == "stress150" else dict()
    p = make_params(batch, n_columns, **kw)
    lp = to_lib_params(p)
    ora = run_oracle(batch, p, n_threads=16, dense=False)
    parts = batch.split_on_start_borders(5)
    assert len(parts) >= 4 and sum(b.n_records for b in parts) == batch.n_records
    dout = engine.alloc_device_outputs(n_columns, lp.mito_length, max(b.n_records for b in parts), overflow_capacity=1 << 16)
    poison(dout)
    engine.stream_begin(lp, dout)
    for b in parts:
        engine.stream_add(b, lp, dout)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = engine.lib.mgatk_stream_finish_device(engine.handle, ctypes.byref(lp), ctypes.byref(engine._outputs_c(dout)), stream)
    assert rc == 0
    torch.cuda.synchronize()
    cols = sample_columns(n_columns, info, ora, 6200)
    res = partial_result(engine, dout, lp, cols)
    assert_global_equal_oracle(res, ora)
    assert_device_planes_consistent(dout, res, ora.cell_qc, lp.mito_length)
    assert_columns_equal_oracle(res, batch, p, cols)


# ---------------------------------------------------------------------------------------------------------------- 6. output completeness through the host entry
def test_host_entry_overwrites_previous_batch(engine):
    """The handle's device buffers are reused by the host entry: a deep batch first, then a sparse one with the same
    n_cells and P where half the columns are empty and some dead. The second result must be the second batch's alone."""
    from oracle.oracle import run_oracle
    n_cells = 64
    deep = sorted_concat([synth_batch(n_cells, 200_000, "atac50", seed=31), pile(70_000, 3000, 5, "ACGTACGTAC" * 2),
                          pile(70_000, 9000, 40, "GGGGGGGGGG" * 2, flag=16)])
    p1 = make_params(deep, n_cells, min_distance_from_end=0)
    r1 = engine.run_host(deep, to_lib_params(p1), overflow_capacity=1 << 16)
    assert r1.stats["n_overflow"] > 0 and r1.planes.max() == 65535
    sparse = synth_batch(n_cells // 2, 20_000, "atac50", seed=32)
    sparse.bc_idx[:] = np.where(sparse.bc_idx >= 0, 2 * sparse.bc_idx + 1, sparse.bc_idx)      # even columns stay empty
    n = run_oracle(sparse, make_params(sparse, n_cells), n_threads=8).cell_qc["n_reads"]
    gate = int(np.median(n[n > 0]))                      # about half the occupied columns fall below the gate
    p2 = make_params(sparse, n_cells, min_reads_per_cell=gate)
    ora = run_oracle(sparse, p2, n_threads=8)
    assert ((n > 0) & (n < gate)).sum() > 0 and (n >= gate).sum() > 0 and (n == 0).sum() >= n_cells // 2
    r2 = engine.run_host(sparse, to_lib_params(p2), overflow_capacity=1 << 16)
    assert r2.stats["n_overflow"] == 0
    assert_result_equals_oracle(r2, ora)
    assert not r2.planes[n < gate].any()


# ---------------------------------------------------------------------------------------------------------------- 7. unaligned bc_idx / flag
def test_unaligned_bc_idx_and_flag(engine):
    """bc_idx 4-byte and flag 2-byte aligned (views at element offset 1): the partition histogram takes its scalar
    loop. Every array keeps its natural element alignment; SrcUser::cell4 (partition.cuh) is the only vector load of a
    batch array and is only taken for 16 / 8-byte aligned bc_idx / flag."""
    import torch
    batch = synth_batch(3000, 150_003, "atac50", seed=41)
    assert batch.n_records % 4 == 3
    p = make_params(batch, 3000)
    lp = to_lib_params(p)
    aligned = engine.upload(batch)
    t = dict(aligned.tensors)
    dev = t["bc_idx"].device
    big_bc = torch.empty(batch.n_records + 1, dtype=torch.int32, device=dev)
    big_bc[1:] = t["bc_idx"]
    big_fl = torch.empty(batch.n_records + 1, dtype=torch.int16, device=dev)
    big_fl[1:] = t["flag"].view(torch.int16)
    t["bc_idx"], t["flag"] = big_bc[1:], big_fl[1:].view(torch.uint16)
    assert t["bc_idx"].data_ptr() % 16 == 4 and t["flag"].data_ptr() % 8 == 2
    moved = DeviceBatch(batch.n_records, aligned.blob_bytes, t)
    results = []
    for db in (aligned, moved):
        dout = run_device_poisoned(engine, batch, lp, dbatch=db)
        results.append(engine.download(dout, lp))
    a, b = results
    np.testing.assert_array_equal(a.planes, b.planes)
    np.testing.assert_array_equal(a.cell_qc, b.cell_qc)
    np.testing.assert_array_equal(a.base_totals, b.base_totals)
    assert a.stats == b.stats
    from oracle.oracle import run_oracle
    assert_result_equals_oracle(b, run_oracle(batch, p, n_threads=8), dense=False)


# ---------------------------------------------------------------------------------------------------------------- 8. blob layout independence
def scatter_blobs(batch, seed):
    """The same records with their blobs in a seeded shuffled order, 16-byte gaps between them."""
    rng = np.random.default_rng(seed)
    units = batch.blob_units()
    perm = rng.permutation(batch.n_records)
    sizes = units[perm] + 1
    starts = np.zeros(batch.n_records, np.int64)
    np.cumsum(sizes[:-1], out=starts[1:])
    off = np.zeros(batch.n_records, np.int64)
    off[perm] = starts + 1
    src16 = batch.blob.view("V16")
    dst16 = np.zeros(int(sizes.sum()) + 1, "V16")
    old = batch.blob_off.astype(np.int64)
    for u in range(int(units.max())):
        m = units > u
        dst16[off[m] + u] = src16[old[m] + u]
    return ReadBatch(pos=batch.pos, tlen=batch.tlen, flag=batch.flag, mapq=batch.mapq, bc_idx=batch.bc_idx, l_seq=batch.l_seq,
                     n_cigar=batch.n_cigar, blob_off=off.astype(np.uint32), blob=dst16.view(np.uint8))


@pytest.mark.parametrize("profile,kw", [("atac50", dict()), ("stress150", dict(max_strand_bias=0.8, min_distance_from_end=10))])
def test_blob_layout_independence(engine, profile, kw):
    from oracle.oracle import run_oracle
    batch = synth_batch(64, 60_000, profile, seed=51)
    shuffled = scatter_blobs(batch, 52)
    assert not np.array_equal(shuffled.blob_off, batch.blob_off)
    for i in (0, 777, batch.n_records - 1):
        assert shuffled.record(i) == batch.record(i)
    p = make_params(batch, 64, **kw)
    lp = to_lib_params(p)
    packed = engine.run_host(batch, lp, overflow_capacity=1 << 16)
    packed = {k: np.copy(getattr(packed, k)) for k in ("planes", "cell_qc", "base_totals")} | {"stats": packed.stats}
    res = engine.run_host(shuffled, lp, overflow_capacity=1 << 16)
    for k in ("planes", "cell_qc", "base_totals"):
        np.testing.assert_array_equal(getattr(res, k), packed[k], err_msg=k)
    assert res.stats == packed["stats"]
    assert_result_equals_oracle(res, run_oracle(batch, p, n_threads=8))


# ---------------------------------------------------------------------------------------------------------------- 9. 16-bit strand-bias filter
def filtered_u16(engine, batch, lp):
    """Raw pileup on the device, then mgatk_filter_strand_bias_device on its planes; planes downloaded."""
    import torch
    from mgatk2_b200._lib import ParamsC
    raw = ParamsC.from_buffer_copy(lp)
    raw.flags = 1
    dout = run_device_poisoned(engine, batch, raw)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = engine.lib.mgatk_filter_strand_bias_device(engine.handle, ctypes.c_void_p(dout.planes.data_ptr()), lp.n_cells,
                                                    lp.mito_length, ctypes.c_double(lp.max_strand_bias), stream)
    assert rc == 0
    torch.cuda.synchronize()
    return engine.download(dout, raw).planes


def assert_planes_equal_oracle_dense(planes, ora, P):
    C = planes.shape[0]
    np.testing.assert_array_equal(planes[:, :8, :P].transpose(0, 2, 1).reshape(C, P, 4, 2), ora.counts)
    np.testing.assert_array_equal(planes[:, 8:10, :P].transpose(0, 2, 1), ora.tn5)
    np.testing.assert_array_equal(planes[:, 10, :P], ora.coverage)
    assert not planes[:, :, P:].any()


@pytest.mark.parametrize("P", [16569, 16299])
@pytest.mark.parametrize("bias", [0.5, 0.8, 0.9999, 1.0])
def test_filter_strand_bias_u16(engine, bias, P):
    from oracle.oracle import run_oracle
    batch = synth_batch(64, 60_000, "atac70", seed=61, mito_length=P)
    p = make_params(batch, 64, max_strand_bias=bias, mito_length=P)
    lp = to_lib_params(p)
    ora = run_oracle(batch, p, n_threads=8)
    assert ora.coverage.max() <= 65535
    planes = filtered_u16(engine, batch, lp)
    assert_planes_equal_oracle_dense(planes, ora, P)
    fused = engine.download(run_device_poisoned(engine, batch, lp), lp)
    np.testing.assert_array_equal(planes, fused.planes)


def test_filter_strand_bias_u16_beyond_grid_cap(engine):
    """70 000 cells: the filter's grid stops at 65 535 cells in y, the cells beyond are reached by its loop."""
    from oracle.oracle import run_oracle
    n_cells, P = 70_000, 64
    batch = synth_batch(n_cells, 400_000, "atac50", seed=62, mito_length=P)
    p = make_params(batch, n_cells, max_strand_bias=0.75, mito_length=P)
    lp = to_lib_params(p)
    ora = run_oracle(batch, p, n_threads=16)
    assert (ora.cell_qc["sum_depth"][65535:] > 0).sum() > 1000
    planes = filtered_u16(engine, batch, lp)
    assert_planes_equal_oracle_dense(planes, ora, P)
