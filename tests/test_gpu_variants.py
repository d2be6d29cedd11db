"""GPU checks of the variant statistics (mgatk_variant_stats_device / mgatk_variant_cells_device, mgatk2_b200/variants.py)
against the numpy restatement in oracle/variants.py.

1. Planes built directly (seeded): a planted reference, clonal variants, low-coverage cells, positions without reads
   (reference N), saturated entries on several cells and planes with their overflow list entries, and one entry of
   exactly 65535 that is not in the list. Outputs are filled with 0xA5 first; integer fields must equal the oracle bit
   for bit, the float sums agree to rtol 1e-9, two runs give the same bytes, and the call decision agrees wherever a
   statistic is not within 1e-9 of its threshold.
2. Through the pileup: a seeded atac50 batch on a 2 000-position contig whose SEQ is rewritten from a planted reference
   with per-clone variants and a 0.5 % substitution rate; one batch, the resident DeviceOutputs and a three-part stream.
3. variant_cells against the exact planes, and a cell-mask subset against the oracle on that subset.
4. The pipeline with and without call_variants: the two files match finalize, every other file is unchanged.
"""
import ctypes
import gzip
import os

import numpy as np
import pytest

from mgatk2_b200.engine import OVERFLOW_DTYPE, PileupResult, pos_pad
from mgatk2_b200.variants import (VARIANT_SUMS_DTYPE, call_mask, call_variants, finalize, read_variant_stats, variant_cells,
                                  variant_sums)
from oracle.variants import oracle_variant_sums, reference_alleles

pytestmark = pytest.mark.gpu

INT_FIELDS = [n for n in VARIANT_SUMS_DTYPE.names if n not in ("dev_sum", "dev_sq")]
FLOAT_FIELDS = ("dev_sum", "dev_sq")


# ---------------------------------------------------------------------------------------------------------------- planes
def planted_planes(C, P, seed):
    """(PileupResult with uint16 planes + overflow list, exact counts [C, P, 4, 2], exact coverage [C, P])."""
    rng = np.random.default_rng(seed)
    ref = rng.integers(0, 4, P)
    depth = rng.integers(0, 40, (C, P), dtype=np.int32)
    depth[rng.random(C) < 0.2] //= 6                                   # low-coverage cells
    counts = ((rng.random((C, P, 4, 2), dtype=np.float32) < 0.05) * rng.integers(1, 4, (C, P, 4, 2), dtype=np.int32)).astype(np.int32)
    fwd = rng.binomial(depth, 0.5).astype(np.int32)
    counts[np.arange(C)[:, None], np.arange(P)[None, :], ref[None, :], 0] += fwd
    counts[np.arange(C)[:, None], np.arange(P)[None, :], ref[None, :], 1] += depth - fwd
    for k in range(min(12, P)):                                        # clonal variants
        p = int(rng.integers(0, P))
        alt = (ref[p] + 1 + k % 3) % 4
        clone = rng.random(C) < 0.3
        counts[clone, p, alt, 0] += rng.integers(2, 15, int(clone.sum()))
        counts[clone, p, alt, 1] += rng.integers(2, 15, int(clone.sum()))
    empty = rng.integers(0, P, max(1, P // 100))                       # reference N
    counts[:, empty] = 0
    for i in range(min(6, C * P)):                                     # saturated entries
        c, p = int(rng.integers(0, C)), int(rng.integers(0, P))
        b, s = int(rng.integers(0, 4)), int(rng.integers(0, 2))
        counts[c, p, b, s] = int(rng.integers(65536, 300000))
    c, p = int(rng.integers(0, C)), int(rng.integers(0, P))
    counts[c, p, ref[p], 0] = 65535 - counts[c, p].sum() + counts[c, p, ref[p], 0]   # coverage exactly 65535, not listed
    cov = counts.sum(axis=(2, 3))
    planes = np.zeros((C, 11, pos_pad(P)), np.uint16)
    ovf = []
    for k in range(8):
        v = counts[:, :, k // 2, k % 2]
        planes[:, k, :P] = np.minimum(v, 65535)
        for cc, pp in zip(*np.nonzero(v > 65535)):
            ovf.append((cc, (k << 24) | pp, v[cc, pp]))
    planes[:, 10, :P] = np.minimum(cov, 65535)
    for cc, pp in zip(*np.nonzero(cov > 65535)):
        ovf.append((cc, (10 << 24) | pp, cov[cc, pp]))
    rng.shuffle(ovf)
    overflow = np.array(ovf, OVERFLOW_DTYPE) if ovf else np.zeros(0, OVERFLOW_DTYPE)
    bt = counts.sum(axis=(0, 3))
    qc = np.zeros(C, [("n_reads", "<u4"), ("n_paired", "<u4"), ("sum_depth", "<u8"), ("covered", "<u4"),
                      ("max_depth", "<u4"), ("median_lo", "<u4"), ("median_hi", "<u4")])
    qc["n_reads"], qc["sum_depth"] = 1, 1
    res = PileupResult(planes, qc, {"n_overflow": len(overflow)}, bt.astype(np.int64), overflow, P)
    assert (planes == 65535).sum() > len(overflow)                     # the unlisted 65535 is there
    return res, counts.astype(np.uint32), cov.astype(np.uint32)


def oracle_chunked(counts, cov, ref, mask=None, low=10, step=2048):
    return np.concatenate([oracle_variant_sums(counts[:, p:p + step], cov[:, p:p + step], ref[p:p + step], mask, low)
                           for p in range(0, cov.shape[1], step)])


def device_sums_poisoned(res, engine, mask=None, low=10):
    """mgatk_variant_stats_device into a 0xA5-filled buffer."""
    import torch

    from mgatk2_b200 import variants
    src = variants._Source(res, engine)
    dev = torch.device("cuda", engine.device)
    out = torch.full((src.mito_length * 4 * VARIANT_SUMS_DTYPE.itemsize,), 0xA5, dtype=torch.uint8, device=dev)
    m = torch.from_numpy(mask.astype(np.uint8)).to(dev) if mask is not None else None
    rc = engine.lib.mgatk_variant_stats_device(engine.handle, ctypes.byref(src.params), ctypes.byref(src.outputs),
                                               m.data_ptr() if m is not None else None, low, out.data_ptr(), src.stream())
    assert rc == 0, engine.lib.mgatk_last_error(engine.handle)
    return out.cpu().numpy().view(VARIANT_SUMS_DTYPE).reshape(src.mito_length, 4)


def assert_sums_equal(got, want):
    for f in INT_FIELDS:
        np.testing.assert_array_equal(got[f], want[f], err_msg=f)
    for f in FLOAT_FIELDS:
        np.testing.assert_allclose(got[f], want[f], rtol=1e-9, atol=1e-15, err_msg=f)
    assert not got["reserved"].any()


def assert_tables_agree(tg, to):
    assert tg["variant"].tolist() == to["variant"].tolist()
    for f in tg.dtype.names:
        if tg.dtype[f].kind == "f":
            np.testing.assert_allclose(tg[f], to[f], rtol=1e-9, atol=1e-15, equal_nan=True, err_msg=f)
        else:
            np.testing.assert_array_equal(tg[f], to[f], err_msg=f)
    near = (np.abs(to["strand_correlation"] - 0.65) < 1e-9) | (np.abs(to["vmr"] - 0.01) < 1e-9)
    np.testing.assert_array_equal(call_mask(tg)[~near], call_mask(to)[~near])


@pytest.fixture(scope="module")
def engine():
    from mgatk2_b200.pileup import get_engine
    return get_engine(0)


@pytest.mark.parametrize("C,P", [(1, 1000), (37, 16569), (2049, 1000), (5000, 1000), (37, 70000), (2049, 16569)])
def test_planes_built_directly(engine, C, P):
    res, counts, cov = planted_planes(C, P, seed=C * 7 + P)
    ref = reference_alleles(res.base_totals)
    assert (ref < 0).any()
    got = device_sums_poisoned(res, engine)
    assert got.tobytes() == device_sums_poisoned(res, engine).tobytes()          # run to run: the same bits
    want = oracle_chunked(counts, cov, ref)
    assert_sums_equal(got, want)
    assert_tables_agree(finalize(got, C), finalize(want, C))
    assert got.tobytes() == variant_sums(res, engine, cells=np.ones(C, bool)).tobytes()


def test_variant_cells_and_cell_mask(engine):
    C, P = 300, 16569
    res, counts, cov = planted_planes(C, P, seed=99)
    sat = res.overflow[(res.overflow["plane_pos"] >> 24) < 8]
    ids = [int(o["plane_pos"] & 0xFFFFFF) * 4 + int(o["plane_pos"] >> 24) // 2 for o in sat]
    ids += [int((res.overflow["plane_pos"][-1] & 0xFFFFFF) * 4), 0, 4 * P - 1, 17 * 4 + 2]
    got = variant_cells(res, np.array(ids, np.int32), engine)
    p, b = np.array(ids) // 4, np.array(ids) % 4
    want = np.stack([counts[:, p, b, 0].T, counts[:, p, b, 1].T, cov[:, p].T], axis=1)
    np.testing.assert_array_equal(got, want)
    assert got.max() > 65535
    mask = np.random.default_rng(1).random(C) < 0.4
    ref = reference_alleles(res.base_totals)
    sub = device_sums_poisoned(res, engine, mask=mask, low=7)
    assert_sums_equal(sub, oracle_chunked(counts, cov, ref, mask, low=7))
    assert_sums_equal(variant_sums(res, engine, cells=np.nonzero(mask)[0], low_coverage_threshold=7), sub)


def test_bad_arguments(engine):
    from mgatk2_b200 import variants
    res, _, _ = planted_planes(3, 100, seed=1)
    src = variants._Source(res, engine)
    lib, h = engine.lib, engine.handle
    assert lib.mgatk_variant_stats_device(h, ctypes.byref(src.params), ctypes.byref(src.outputs), None, 0, 1, None) == 1
    assert lib.mgatk_variant_stats_device(h, ctypes.byref(src.params), ctypes.byref(src.outputs), None, 10, None, None) == 1
    assert lib.mgatk_variant_cells_device(h, ctypes.byref(src.params), ctypes.byref(src.outputs), None, -1, None, None) == 1
    big = type(src.params).from_buffer_copy(src.params)
    big.mito_length = 1 << 24
    assert lib.mgatk_variant_stats_device(h, ctypes.byref(big), ctypes.byref(src.outputs), None, 10, 1, None) == 8
    assert b"mito_length" in lib.mgatk_last_error(h)
    with pytest.raises(ValueError):
        variant_cells(res, np.array([400], np.int32), engine)


# ---------------------------------------------------------------------------------------------------------------- pileup
P_SHORT = 2000
CLONES = {0: [(301, 2), (777, 1), (1500, 3)], 1: [(420, 1), (1234, 2)], 2: [(950, 3), (1800, 1)]}   # pos, alt - ref (mod 4)


def planted_batch(n_cells=96, n_records=300_000, seed=4242):
    """atac50 batch whose SEQ follows a planted reference, with the variants of CLONES in the cells of clone c % 4
    (clone 3: none) and a 0.5 % substitution rate. Returns (batch, reference, planted variant names)."""
    from mgatk2_b200.synth import synth_batch
    batch = synth_batch(n_cells, n_records, "atac50", seed=seed, mito_length=P_SHORT)
    rng = np.random.default_rng(seed + 1)
    ref = rng.integers(0, 4, P_SHORT + 64)
    assert (batch.n_cigar == 1).all() and (batch.l_seq == 50).all()
    n, L = batch.n_records, 50
    at = batch.pos[:, None].astype(np.int64) + np.arange(L)[None, :]
    base = ref[np.minimum(at, len(ref) - 1)]
    cell = np.where(batch.bc_idx >= 0, batch.bc_idx, -1)
    planted = []
    for clone, variants in CLONES.items():
        in_clone = (cell >= 0) & (cell % 4 == clone)
        for p, off in variants:
            alt = (ref[p] + off) % 4
            base = np.where(in_clone[:, None] & (at == p), alt, base)
            planted.append(f"{p + 1}{'ACGT'[ref[p]]}>{'ACGT'[alt]}")
    sub = rng.random((n, L)) < 0.005
    base = np.where(sub, (base + rng.integers(1, 4, (n, L))) % 4, base)
    code = np.array([1, 2, 4, 8], np.uint8)[base]
    packed = (code[:, 0::2] << 4) | code[:, 1::2]
    start = batch.blob_off.astype(np.int64) * 16 + 4
    blob = batch.blob.copy()
    blob[start[:, None] + np.arange(L // 2)[None, :]] = packed
    batch.blob = blob
    return batch, ref[:P_SHORT], sorted(planted)


@pytest.fixture(scope="module")
def planted():
    from oracle.oracle import make_params, run_oracle
    batch, ref, names = planted_batch()
    params = make_params(96, mito_length=P_SHORT, max_read_extent=batch.max_read_extent())
    ora = run_oracle(batch, params, n_threads=8)
    return batch, params, ora, names


def oracle_of(ora, min_reads=1):
    n = ora.cell_qc["n_reads"].astype(np.int64)
    alive = (n >= max(1, min_reads)) & (ora.cell_qc["sum_depth"] > 0)
    sums = oracle_variant_sums(ora.counts, ora.coverage, reference_alleles(ora.base_totals), alive)
    return sums, int(alive.sum())


def test_through_the_pileup(engine, planted):
    import torch

    from mgatk2_b200._lib import ParamsC
    batch, params, ora, names = planted
    want, n = oracle_of(ora)
    t_want = finalize(want, n)
    assert sorted(call_variants(t_want)["variant"].tolist()) == names
    lp = ParamsC(*[getattr(params, f) for f, _ in params._fields_])
    res = engine.run_host(batch, lp)
    got = variant_sums(res, engine)
    assert_sums_equal(got, want)
    assert sorted(call_variants(finalize(got, n))["variant"].tolist()) == names
    # resident outputs: nothing downloaded
    dout = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    engine.run_device(engine.upload(batch), lp, dout)
    got_dev = variant_sums((dout, lp), engine)
    assert got_dev.tobytes() == got.tobytes()
    # three parts through the resident planes
    dout_s = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    res_s = engine.run_stream(batch.split_on_start_borders(3), lp, dout_s)
    assert_sums_equal(variant_sums((dout_s, lp), engine), want)
    assert_sums_equal(variant_sums(res_s, engine), want)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- pipeline
def _files(root):
    out = {}
    for dirpath, _, files in os.walk(root):
        for f in files:
            out[os.path.relpath(os.path.join(dirpath, f), root)] = open(os.path.join(dirpath, f), "rb").read()
    return out


def _summary_body(b):
    return [line for line in b.decode().splitlines() if not line.startswith(("run_date", "output_dir"))]


@pytest.mark.parametrize("fmt", ["standard", "hdf5"])
def test_pipeline_call_variants(engine, planted, tmp_path, fmt):
    from mgatk2_b200 import BAMReader, PipelineConfig, run_pipeline
    from mgatk2_b200.bamio import write_bam
    from mgatk2_b200.barcodes import load_barcodes
    from mgatk2_b200.synth import make_whitelist
    batch, _, _, names = planted
    barcodes = make_whitelist(96, seed=3)
    bam = str(tmp_path / "possorted_bam.bam")
    write_bam(bam, batch, barcodes, ref_lens=(248956422, P_SHORT, 156040895), write_index=False)
    kw = dict(barcode_file=None, min_barcode_reads=10, output_format=fmt, mito_length=P_SHORT, max_strand_bias=1.0)
    run_pipeline(bam, str(tmp_path / "plain"), **kw)
    run_pipeline(bam, str(tmp_path / "called"), call_variants=True, **kw)
    plain, called = _files(tmp_path / "plain"), _files(tmp_path / "called")
    extra = {"output/variant_stats.tsv.gz", "output/variant_cells.tsv.gz"}
    assert set(called) == set(plain) | extra
    for k in plain:
        if k == "qc/summary.txt":
            assert _summary_body(plain[k]) == _summary_body(called[k])
        else:
            assert plain[k] == called[k], k
    # the files against finalize of the seam's own result
    wl, _ = load_barcodes(None, bam, barcode_tag="CB", mito_chr="chrM", min_barcode_reads=10)
    cfg = PipelineConfig(mito_length=P_SHORT, max_strand_bias=1.0)
    rbb, _ = BAMReader(bam, cfg, set(wl), barcode_list=list(wl)).collect_reads_by_barcode()
    res = rbb.result
    alive = res.alive()
    table = finalize(variant_sums(res, engine), int(alive.sum()))
    back = read_variant_stats(tmp_path / "called" / "output" / "variant_stats.tsv.gz")
    assert back["variant"].tolist() == table["variant"].tolist()
    for f in table.dtype.names:
        if table.dtype[f].kind == "f":
            np.testing.assert_allclose(back[f], table[f], rtol=1e-9, atol=1e-15, equal_nan=True, err_msg=f)
        else:
            np.testing.assert_array_equal(back[f], table[f], err_msg=f)
    hits = call_variants(table)
    assert sorted(hits["variant"].tolist()) == names
    counts = variant_cells(res, hits, engine)
    cols = res.columns if res.columns is not None else np.arange(len(res.planes))
    want = ["variant\tbarcode\talt_fwd\talt_rev\tcoverage"]
    for i, name in enumerate(hits["variant"].tolist()):
        f, r, d = counts[i]
        want += [f"{name}\t{wl[int(cols[k])]}\t{f[k]}\t{r[k]}\t{d[k]}" for k in range(len(cols)) if alive[k] and d[k] > 0]
    got = gzip.open(tmp_path / "called" / "output" / "variant_cells.tsv.gz", "rt").read().splitlines()
    assert got == want and len(got) > len(names)
