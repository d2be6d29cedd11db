"""GPU checks of the clone markers (mgatk_marker_ranks_device, mgatk2_b200/markers.py) against the numpy restatement in
oracle/markers.py.

1. Counts built directly (planted_counts of test_gpu_clones.py) with equal x from different (a, d), neighbours one ulp
   apart, d = 0 cells, labels 0, negative and above G, empty groups and everything in one group; variants with exactly
   kMarkerS and kMarkerS + 1 nonzero values and one with every population cell nonzero (the shared-memory sort and the
   merge fallback), G on both sides of kMarkerGs. rank2 and ties equal the oracle exactly, outputs filled with 0xA5
   first, two calls give the same bytes.
2. Bad arguments return the documented status codes.
3. Through the pileup: the planted four-clone batch of test_gpu_variants.py, one batch, the resident DeviceOutputs and a
   three-part stream; find_clones then clone_markers against the oracle on the oracle's planes, and each planted clone's
   variants have smaller p values in its clone than every other variant.
4. The pipeline with clone_markers: one more file, equal to clone_markers of the same result, every other file as with
   find_clones; a run without called variants writes the header alone.
"""
import ctypes
import gzip
import re
from fractions import Fraction

import numpy as np
import pytest

from oracle import clones as oc
from oracle import markers as om
from tests.test_gpu_clones import planted_counts
from tests.test_gpu_variants import CLONES, P_SHORT, _files, _summary_body, oracle_of, planted_batch

pytestmark = pytest.mark.gpu

S = 4096                                    # kMarkerS
G_S = 1024                                  # kMarkerGs


@pytest.fixture(scope="module")
def engine():
    from mgatk2_b200.pileup import get_engine
    return get_engine(0)


def device_ranks(engine, counts, labels, G, fill=0xA5):
    import torch
    dev = torch.device("cuda", engine.device)
    V, _, C = counts.shape
    c_t = torch.from_numpy(counts.view(np.int32).copy()).to(dev)
    l_t = torch.from_numpy(np.ascontiguousarray(labels, np.int32)).to(dev)
    rank2 = torch.full((V * G * 8,), fill, dtype=torch.uint8, device=dev)
    ties = torch.full((V * 8,), fill, dtype=torch.uint8, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    lib, h = engine.lib, engine.handle
    rc = lib.mgatk_marker_ranks_device(h, c_t.data_ptr(), l_t.data_ptr(), C, V, G, rank2.data_ptr(), ties.data_ptr(),
                                       stream)
    assert rc == 0, lib.mgatk_last_error(h)
    return rank2.cpu().numpy().view(np.uint64).reshape(V, G), ties.cpu().numpy().view(np.uint64)


def ulp_pair():
    """((a1, d1), (a2, d2)) whose x are neighbours in fp64: a2 / d2 is the best fraction with d2 < 2^32 for the double
    one ulp above a1 / d1."""
    a1, d1 = 1234567891, 3456789013
    up = np.nextafter(np.float64(a1) / np.float64(d1), 1.0)
    f = Fraction(float(up)).limit_denominator(2 ** 32 - 1)
    assert np.float64(f.numerator) / np.float64(f.denominator) == up
    return (a1, d1), (f.numerator, f.denominator)


def marker_counts(C, V, G, seed, big=False):
    """planted_counts with the planted ties and neighbours, and labels with every kind of excluded cell."""
    rng = np.random.default_rng(seed)
    counts = planted_counts(C, V, seed).astype(np.uint64)
    labels = rng.integers(1, G + 1, C).astype(np.int64)
    if G >= 3:
        labels[labels == 2] = 3                                                 # group 2 empty
    labels[rng.random(C) < 0.05] = 0
    labels[rng.random(C) < 0.03] = -7
    labels[rng.random(C) < 0.03] = G + 1 + rng.integers(0, 5, C)[0]
    (a_lo, d_lo), (a_up, d_up) = ulp_pair()
    for v in range(V):
        cells = rng.choice(C, min(C, 12), replace=False)
        for j, c in enumerate(cells):
            kind = j % 4
            if kind == 0:                                                       # 1/2 = 2/4 = 3/6
                k = 1 + j % 3
                counts[v, :, c] = (k, 0, 2 * k)
            elif kind == 1:                                                     # one ulp apart
                counts[v, :, c] = (a_lo, 0, d_lo)
            elif kind == 2:
                counts[v, :, c] = (a_up, 0, d_up)
            else:                                                               # detected, not covered: x = 0
                counts[v, :, c] = (4, 1, 0)
    if big:
        inside = np.flatnonzero((labels >= 1) & (labels <= G))
        dense = rng.integers(1, 40, (3, C)).astype(np.uint64)
        for v, n_hit in zip(range(min(V, 4)), [S, S + 1, 2 * S + 3, len(inside)]):
            counts[v] = 0
            counts[v, 2] = dense[v % 3]
            hit = rng.choice(inside, n_hit, replace=False)
            counts[v, 0, hit] = rng.integers(1, 4, n_hit)
            counts[v, 2, hit] = np.maximum(counts[v, 2, hit], counts[v, 0, hit])
    return counts.astype(np.uint32), labels.astype(np.int32)


@pytest.mark.parametrize("C,V,G", [(1, 3, 1), (37, 5, 2), (400, 9, 7), (2000, 64, 7), (9000, 12, 1), (12000, 300, 2),
                                   (20000, 6, 1500), (50000, 8, 7), (50000, 5, 2000)])
def test_ranks_exact(engine, C, V, G):
    counts, labels = marker_counts(C, V, G, seed=C + V + G, big=C >= 12000)
    want_r2, want_ties = om.marker_ranks(counts, labels, G)
    r2, ties = device_ranks(engine, counts, labels, G)
    np.testing.assert_array_equal(r2, want_r2)
    np.testing.assert_array_equal(ties, want_ties)
    r2b, tiesb = device_ranks(engine, counts, labels, G, fill=0x5A)
    assert r2b.tobytes() == r2.tobytes() and tiesb.tobytes() == ties.tobytes()
    if C >= 12000:                                                             # both sort paths were taken
        x = oc.allele_frequencies(counts)
        inside = (labels >= 1) & (labels <= G)
        nnz = (x[:, inside] > 0).sum(axis=1)
        assert nnz[0] == S and nnz[1] == S + 1 and nnz[2] == 2 * S + 3 and nnz[3] == inside.sum()


def test_one_group_and_no_population(engine):
    counts, _ = marker_counts(3000, 7, 1, seed=5)
    every = np.ones(3000, np.int32)                                             # the rest is empty
    want = om.marker_ranks(counts, every, 1)
    got = device_ranks(engine, counts, every, 1)
    np.testing.assert_array_equal(got[0], want[0])
    np.testing.assert_array_equal(got[1], want[1])
    assert (got[0][:, 0] == 3000 * 3001).all()                                  # 2 * (1 + ... + N)
    none = np.zeros(3000, np.int32)                                            # nobody in the test: zeros
    r2, ties = device_ranks(engine, counts, none, 4)
    assert not r2.any() and not ties.any()


def test_bad_arguments(engine, monkeypatch):
    import torch
    lib, h = engine.lib, engine.handle
    dev = torch.device("cuda", engine.device)
    buf = torch.zeros(1 << 16, dtype=torch.int64, device=dev)
    p = buf.data_ptr()
    ok = dict(counts=p, labels=p, C=8, V=3, G=2, r2=p, ties=p)

    def call(**kw):
        a = dict(ok, **kw)
        return lib.mgatk_marker_ranks_device(h, a["counts"], a["labels"], a["C"], a["V"], a["G"], a["r2"], a["ties"], None)
    assert call(C=-1) == 1 and call(V=-1) == 1 and call(G=0) == 1 and call(G=-3) == 1
    assert call(counts=None) == 1 and call(labels=None) == 1 and call(r2=None) == 1 and call(ties=None) == 1
    assert call(C=(1 << 21) + 1) == 8 and call(V=4097) == 8 and call(G=9) == 8
    assert call(V=0, counts=None, r2=None, ties=None) == 0
    assert call(C=0, counts=None, labels=None, G=5) == 0
    torch.cuda.synchronize()
    assert not buf[: 3 * 5].any()                                               # n_cells = 0: zero outputs
    buf.fill_(7)
    assert call(C=0, counts=None, labels=None, G=2) == 0
    torch.cuda.synchronize()
    assert not buf[: 3 * 2].any()
    from mgatk2_b200.exceptions import ProcessingError
    from mgatk2_b200.markers import find_markers
    from mgatk2_b200.variants import _Source
    res = planted_result()
    src = _Source(res, engine)
    with pytest.raises(ValueError):
        find_markers(src, np.ones(5, np.int32), [0])
    with pytest.raises(ValueError):
        find_markers(src, np.full(src.n_cells, src.n_cells + 1, np.int32), [0])
    monkeypatch.setattr("mgatk2_b200.markers.MAX_CELLS", 10)                   # 20 cells in the test: refused
    with pytest.raises(ProcessingError):
        find_markers(src, np.ones(src.n_cells, np.int32), [0])


def planted_result():
    """A small host result for the argument checks."""
    from mgatk2_b200.engine import PileupResult, pos_pad
    C, P = 20, 100
    planes = np.zeros((C, 11, pos_pad(P)), np.uint16)
    qc = np.zeros(C, [("n_reads", "<u4"), ("n_paired", "<u4"), ("sum_depth", "<u8"), ("covered", "<u4"),
                      ("max_depth", "<u4"), ("median_lo", "<u4"), ("median_hi", "<u4")])
    qc["n_reads"], qc["sum_depth"] = 1, 1
    from mgatk2_b200.engine import OVERFLOW_DTYPE
    return PileupResult(planes, qc, {"n_overflow": 0}, np.zeros((P, 4), np.int64), np.zeros(0, OVERFLOW_DTYPE), P)


# ---------------------------------------------------------------------------------------------------------------- pileup
@pytest.fixture(scope="module")
def planted():
    from oracle.oracle import make_params, run_oracle
    batch, ref, names = planted_batch()
    params = make_params(96, mito_length=P_SHORT, max_read_extent=batch.max_read_extent())
    ora = run_oracle(batch, params, n_threads=8)
    return batch, params, ora, names


def oracle_markers(ora):
    """(labels, rank2, ties, counts) of the oracle's planes: clones by oracle/clones.py, ranks by oracle/markers.py."""
    from mgatk2_b200.variants import call_variants, finalize, variant_ids
    sums, n = oracle_of(ora)
    called = call_variants(finalize(sums, n))
    ids = variant_ids(called)
    p, b = ids // 4, ids % 4
    counts = np.stack([ora.counts[:, p, b, 0].T, ora.counts[:, p, b, 1].T, ora.coverage[:, p].T], axis=1).astype(np.uint32)
    nr = ora.cell_qc["n_reads"].astype(np.int64)
    alive = (nr >= 1) & (ora.cell_qc["sum_depth"] > 0)
    labels, _ = oc.oracle_find_clones(counts, alive)
    G = int(labels.max())
    rank2, ties = om.marker_ranks(counts, labels, G)
    return labels, rank2, ties, counts, called


def test_through_the_pileup(engine, planted):
    import torch

    from mgatk2_b200._lib import ParamsC
    from mgatk2_b200.clones import find_clones
    from mgatk2_b200.markers import clone_markers, wilcoxon
    batch, params, ora, names = planted
    labels, rank2, ties, counts, called = oracle_markers(ora)
    G, V = int(labels.max()), len(called)
    lp = ParamsC(*[getattr(params, f) for f, _ in params._fields_])
    res = engine.run_host(batch, lp)
    clones = find_clones(res, engine=engine)
    np.testing.assert_array_equal(clones.labels, labels)
    got = clone_markers(res, clones, engine)
    assert len(got) == G * V
    N = int((labels > 0).sum())
    for g in range(1, G + 1):
        n1 = int((labels == g).sum())
        for v in range(V):
            row = got[(g - 1) * V + v]
            assert row["clone"] == g and row["variant"] == clones.variant_names[v]
            U, auc, _, p = wilcoxon(rank2[v, g - 1], ties[v], n1, N)
            assert row["statistic"] == U and row["n_cells"] == n1 and row["n_cells_rest"] == N - n1
            np.testing.assert_array_equal([row["auc"], row["p_value"]], [auc, p])
    # the same table from the resident outputs and from a three-part stream
    dout = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    engine.run_device(engine.upload(batch), lp, dout)
    assert clone_markers((dout, lp), clones, engine).tobytes() == got.tobytes()
    dout_s = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    res_s = engine.run_stream(batch.split_on_start_borders(3), lp, dout_s)
    assert clone_markers((dout_s, lp), clones, engine).tobytes() == got.tobytes()
    assert clone_markers(res_s, clones, engine).tobytes() == got.tobytes()
    # each planted clone's variants come before every other variant of its clone by p value
    cells = np.arange(96)
    for q, planted_vars in CLONES.items():
        lab = labels[(cells % 4 == q) & (labels > 0)]
        k = int(np.bincount(lab).argmax())
        rows = got[got["clone"] == k]
        mine = np.array([int(re.match(r"\d+", v).group()) in {p + 1 for p, _ in planted_vars} for v in rows["variant"]])
        assert mine.sum() == len(planted_vars)
        assert rows["p_value"][mine].max() < rows["p_value"][~mine].min(), (q, rows[["variant", "p_value"]])
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- pipeline
def test_pipeline_clone_markers(engine, planted, tmp_path):
    from mgatk2_b200 import BAMReader, PipelineConfig, run_pipeline
    from mgatk2_b200.bamio import write_bam
    from mgatk2_b200.barcodes import load_barcodes
    from mgatk2_b200.clones import find_clones
    from mgatk2_b200.markers import clone_markers, write_clone_markers
    from mgatk2_b200.synth import make_whitelist
    batch, _, _, _ = planted
    barcodes = make_whitelist(96, seed=3)
    bam = str(tmp_path / "possorted_bam.bam")
    write_bam(bam, batch, barcodes, ref_lens=(248956422, P_SHORT, 156040895), write_index=False)
    kw = dict(barcode_file=None, min_barcode_reads=10, mito_length=P_SHORT, max_strand_bias=1.0)
    run_pipeline(bam, str(tmp_path / "clones"), find_clones=True, **kw)
    run_pipeline(bam, str(tmp_path / "markers"), clone_markers=True, **kw)
    base, got = _files(tmp_path / "clones"), _files(tmp_path / "markers")
    assert set(got) == set(base) | {"output/clone_markers.tsv.gz"}
    for k in base:
        if k == "qc/summary.txt":
            assert _summary_body(base[k]) == _summary_body(got[k])
        else:
            assert base[k] == got[k], k
    wl, _ = load_barcodes(None, bam, barcode_tag="CB", mito_chr="chrM", min_barcode_reads=10)
    cfg = PipelineConfig(mito_length=P_SHORT, max_strand_bias=1.0)
    rbb, _ = BAMReader(bam, cfg, set(wl), barcode_list=list(wl)).collect_reads_by_barcode()
    clones = find_clones(rbb.result, engine=engine)
    table = clone_markers(rbb.result, clones, engine)
    assert clones.n_clones >= 3 and len(table) == clones.n_clones * len(clones.variants)
    (tmp_path / "want").mkdir()
    write_clone_markers(table, tmp_path / "want" / "clone_markers.tsv.gz")      # gzip keeps the file name
    assert got["output/clone_markers.tsv.gz"] == (tmp_path / "want" / "clone_markers.tsv.gz").read_bytes()
    # too few reads for any variant to be called: the file holds its header alone
    sparse, _, _ = planted_batch(n_records=3000, seed=77)
    bam2 = str(tmp_path / "sparse.bam")
    write_bam(bam2, sparse, barcodes, ref_lens=(248956422, P_SHORT, 156040895), write_index=False)
    run_pipeline(bam2, str(tmp_path / "sparse"), clone_markers=True, **dict(kw, min_barcode_reads=1))
    assert gzip.open(tmp_path / "sparse" / "output" / "variant_cells.tsv.gz", "rt").read().count("\n") == 1
    text = gzip.open(tmp_path / "sparse" / "output" / "clone_markers.tsv.gz", "rt").read()
    assert text.count("\n") == 1 and text.startswith("clone\tvariant\t")
