"""GPU checks of the clone step (mgatk_clone_knn_device / mgatk_clone_snn_device, mgatk2_b200/clones.py) against the
numpy restatement in oracle/clones.py.

1. Counts built directly (seeded, clone-structured) with planted exact duplicates (the same counts, and counts scaled
   with the coverage so x is equal) and rows that differ from another only in the last bits (x scaled by 3 or 5): the kNN
   lists and similarities equal the oracle bit for bit, outputs filled with 0xA5 first, two calls give the same bytes;
   the SNN weights equal the oracle's exactly.
2. Bad arguments return the documented status codes.
3. Through the pileup: the planted four-clone batch of test_gpu_variants.py, one batch, the resident DeviceOutputs and a
   three-part stream, against the oracle run on the oracle's planes.
4. The pipeline with find_clones: two more files, every other file unchanged.
"""
import ctypes
import os

import numpy as np
import pytest

from oracle import clones as oc
from tests.test_gpu_variants import P_SHORT, _files, _summary_body, oracle_of, planted_batch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from mgatk2_b200.pileup import get_engine
    return get_engine(0)


def planted_counts(C, V, seed):
    """uint32 [V, 3, C]: cells in a few clones, noise, cells without any detection, exact duplicates and rows whose x is
    another row's times 2, 3 or 5."""
    rng = np.random.default_rng(seed)
    d = rng.integers(1, 60, (V, C)).astype(np.uint64)
    d[rng.random((V, C)) < 0.1] = 0
    het = np.where(rng.random((V, C)) < 0.05, rng.random((V, C)) * 0.2, 0.0)
    n_clones = 4
    clone = rng.integers(0, n_clones, C)
    for q in range(n_clones):
        for v in range(q % V, V, n_clones):
            m = clone == q
            het[v, m] = rng.uniform(0.2, 0.95, int(m.sum()))
    a = np.floor(het * d).astype(np.uint64)
    f = rng.binomial(a.astype(np.int64), 0.5).astype(np.uint64)
    r = a - f
    if C > 1:
        for t in range(max(1, C // 10)):
            src, dst = int(rng.integers(0, C)), int(rng.integers(0, C))
            kind = t % 4
            if kind == 0:                                   # exact duplicate
                f[:, dst], r[:, dst], d[:, dst] = f[:, src], r[:, src], d[:, src]
            elif kind == 1:                                 # x equal: counts and coverage doubled
                f[:, dst], r[:, dst], d[:, dst] = 2 * f[:, src], 2 * r[:, src], 2 * d[:, src]
            else:                                           # x * 3 or x * 5: the same direction up to rounding
                m = 3 if kind == 2 else 5
                f[:, dst], r[:, dst], d[:, dst] = m * f[:, src], m * r[:, src], d[:, src]
    empty = rng.random(C) < 0.05
    f[:, empty] = 0
    r[:, empty] = 0
    return np.stack([f, r, d], axis=1).astype(np.uint32)


def device_knn(engine, counts, rows, k, fill=0xA5):
    import torch
    dev = torch.device("cuda", engine.device)
    V, _, C = counts.shape
    n = len(rows)
    k_eff = min(k, n)
    c_t = torch.from_numpy(counts.view(np.int32).copy()).to(dev)
    r_t = torch.from_numpy(rows.astype(np.int32)).to(dev)
    nbr = torch.full((n * k_eff * 4,), fill, dtype=torch.uint8, device=dev)
    sim = torch.full((n * k_eff * 8,), fill, dtype=torch.uint8, device=dev)
    w = torch.full((n * k_eff * 8,), fill, dtype=torch.uint8, device=dev)
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    lib, h = engine.lib, engine.handle
    rc = lib.mgatk_clone_knn_device(h, c_t.data_ptr(), r_t.data_ptr(), n, C, V, k, nbr.data_ptr(), sim.data_ptr(), stream)
    assert rc == 0, lib.mgatk_last_error(h)
    rc = lib.mgatk_clone_snn_device(h, nbr.data_ptr(), n, k_eff, w.data_ptr(), stream)
    assert rc == 0, lib.mgatk_last_error(h)
    return (nbr.cpu().numpy().view(np.int32).reshape(n, k_eff), sim.cpu().numpy().view(np.float64).reshape(n, k_eff),
            w.cpu().numpy().view(np.float64).reshape(n, k_eff))


@pytest.mark.parametrize("n_cells,V,k", [(1, 7, 10), (5, 1, 2), (6, 7, 64), (300, 64, 33), (300, 1, 10), (777, 7, 64),
                                         (2500, 200, 10), (2500, 64, 64), (2531, 7, 2), (1000, 200, 33)])
def test_knn_and_snn_bit_exact(engine, n_cells, V, k):
    counts = planted_counts(n_cells, V, seed=n_cells * 3 + V + k)
    x = oc.allele_frequencies(counts)
    rows = oc.graph_rows(x)
    if n_cells == 1:
        rows = np.array([0], np.int32)
        counts[:, :, 0] = (1, 1, 3)
        x = oc.allele_frequencies(counts)
    assert len(rows) >= 1
    want_nbr, want_sim = oc.knn(np.ascontiguousarray(x[:, rows].T), k)
    nbr, sim, w = device_knn(engine, counts, rows, k)
    np.testing.assert_array_equal(nbr, want_nbr)
    assert sim.tobytes() == want_sim.tobytes()
    assert w.tobytes() == oc.snn_weights(want_nbr).tobytes()
    nbr2, sim2, w2 = device_knn(engine, counts, rows, k, fill=0x5A)
    assert nbr2.tobytes() == nbr.tobytes() and sim2.tobytes() == sim.tobytes() and w2.tobytes() == w.tobytes()
    if len(rows) > 20:                                      # the planted near-duplicates give ties and last-bit orders
        assert (want_sim[:, 1:] >= 1.0 - 1e-12).any()


def test_rows_without_a_detection(engine):
    """A row that breaks the graph-row rule (no detection, or a cell index outside [0, n_cells)) reads as zeros, gets
    inv = 0 and cosine 0 with every row: the lists stay the oracle's, bit for bit, on every call."""
    counts = planted_counts(400, 9, seed=77)
    x = oc.allele_frequencies(counts)
    empty = np.nonzero(~(x > 0).any(axis=0))[0]
    assert len(empty)
    rows = np.concatenate([oc.graph_rows(x)[:150], empty[:2], [400, -3]]).astype(np.int32)
    rows.sort()
    xr = np.zeros((len(rows), x.shape[0]))
    inside = (rows >= 0) & (rows < 400)
    xr[inside] = x[:, rows[inside]].T
    want_nbr, want_sim = oc.knn(xr, 12)
    assert np.isfinite(want_sim).all()
    nbr, sim, w = device_knn(engine, counts, rows, 12)
    np.testing.assert_array_equal(nbr, want_nbr)
    assert sim.tobytes() == want_sim.tobytes()
    nbr2, sim2, _ = device_knn(engine, counts, rows, 12, fill=0x5A)
    assert nbr2.tobytes() == nbr.tobytes() and sim2.tobytes() == sim.tobytes()


def test_destroy_frees_the_search_scratch():
    """The x / inv scratch of a search (here 20 000 rows x 1 024 padded variants, 164 MB) goes with its handle."""
    import torch

    from mgatk2_b200.engine import PileupEngine
    dev = torch.device("cuda", 0)
    n, V = 20_000, 1000

    def one_search():
        eng = PileupEngine(0)
        g = torch.Generator(device=dev).manual_seed(5)
        counts = torch.randint(1, 9, (V, 3, n), generator=g, device=dev, dtype=torch.int32)
        rows = torch.arange(n, dtype=torch.int32, device=dev)
        nbr = torch.empty((n, 2), dtype=torch.int32, device=dev)
        sim = torch.empty((n, 2), dtype=torch.float64, device=dev)
        s = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        rc = eng.lib.mgatk_clone_knn_device(eng.handle, counts.data_ptr(), rows.data_ptr(), n, n, V, 2, nbr.data_ptr(),
                                            sim.data_ptr(), s)
        assert rc == 0, eng.lib.mgatk_last_error(eng.handle)
        torch.cuda.synchronize()
        eng.close()

    one_search()                                    # first use: module load, torch allocator, context growth
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(3):
        one_search()
    torch.cuda.empty_cache()
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free0 - free1 < 64 << 20, (free0 - free1) >> 20


def test_bad_arguments(engine):
    import torch
    lib, h = engine.lib, engine.handle
    dev = torch.device("cuda", engine.device)
    buf = torch.zeros(1 << 16, dtype=torch.int32, device=dev)
    p = buf.data_ptr()
    ok = dict(counts=p, rows=p, n=4, C=8, V=3, k=3, nbr=p, sim=p)

    def knn(**kw):
        a = dict(ok, **kw)
        return lib.mgatk_clone_knn_device(h, a["counts"], a["rows"], a["n"], a["C"], a["V"], a["k"], a["nbr"], a["sim"], None)
    assert knn(k=1) == 1 and knn(n=-1) == 1 and knn(C=-1) == 1 and knn(V=-1) == 1
    assert knn(k=65) == 1 and b"k must be" in lib.mgatk_last_error(h)
    assert knn(rows=None) == 1 and knn(nbr=None) == 1 and knn(sim=None) == 1 and knn(counts=None) == 1
    assert knn(V=0) == 1 and knn(n=9) == 1
    assert knn(V=4097) == 8
    assert knn(n=(1 << 24) + 1, C=(1 << 24) + 1) == 8
    assert knn(n=1 << 24, C=1 << 24, V=4096) == 8                     # 2^24 rows x 4096 variants: beyond the scratch
    assert knn(n=0, rows=None, nbr=None, sim=None, counts=None) == 0
    torch.cuda.synchronize()
    snn = lib.mgatk_clone_snn_device
    assert snn(h, p, -1, 2, p, None) == 1 and snn(h, p, 4, 0, p, None) == 1 and snn(h, p, 4, 5, p, None) == 1
    assert snn(h, p, 4, 65, p, None) == 1 and snn(h, None, 4, 2, p, None) == 1 and snn(h, p, 4, 2, None, None) == 1
    assert snn(h, p, 0, 2, None, None) == 0
    with pytest.raises(ValueError):
        from mgatk2_b200.clones import find_clones
        find_clones(None, k=65)


# ---------------------------------------------------------------------------------------------------------------- pileup
@pytest.fixture(scope="module")
def planted():
    from oracle.oracle import make_params, run_oracle
    batch, ref, names = planted_batch()
    params = make_params(96, mito_length=P_SHORT, max_read_extent=batch.max_read_extent())
    ora = run_oracle(batch, params, n_threads=8)
    return batch, params, ora, names


def oracle_clones(ora):
    from mgatk2_b200.variants import call_variants, finalize, variant_ids
    sums, n = oracle_of(ora)
    called = call_variants(finalize(sums, n))
    ids = variant_ids(called)
    p, b = ids // 4, ids % 4
    counts = np.stack([ora.counts[:, p, b, 0].T, ora.counts[:, p, b, 1].T, ora.coverage[:, p].T], axis=1).astype(np.uint32)
    nr = ora.cell_qc["n_reads"].astype(np.int64)
    alive = (nr >= 1) & (ora.cell_qc["sum_depth"] > 0)
    return oc.oracle_find_clones(counts, alive), counts, called


def test_through_the_pileup(engine, planted):
    import torch

    from mgatk2_b200._lib import ParamsC
    from mgatk2_b200.clones import allele_frequencies, clone_variants, find_clones
    batch, params, ora, names = planted
    (want, info), counts, called = oracle_clones(ora)
    assert sorted(called["variant"].tolist()) == names
    lp = ParamsC(*[getattr(params, f) for f, _ in params._fields_])
    res = engine.run_host(batch, lp)
    got = find_clones(res, engine=engine)
    np.testing.assert_array_equal(got.labels, want)
    np.testing.assert_array_equal(got.rows, info["rows"])
    np.testing.assert_array_equal(got.neighbors, info["nbr"])
    assert got.similarity.tobytes() == info["sim"].tobytes()
    for a, b in zip((got.indptr, got.indices, got.weights), info["csr"]):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(allele_frequencies(res, called, engine), oc.allele_frequencies(counts))
    dout = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    engine.run_device(engine.upload(batch), lp, dout)
    np.testing.assert_array_equal(find_clones((dout, lp), engine=engine).labels, want)
    dout_s = engine.alloc_device_outputs(96, P_SHORT, batch.n_records, max_read_extent=batch.max_read_extent())
    res_s = engine.run_stream(batch.split_on_start_borders(3), lp, dout_s)
    np.testing.assert_array_equal(find_clones((dout_s, lp), engine=engine).labels, want)
    np.testing.assert_array_equal(find_clones(res_s, engine=engine).labels, want)
    # the planted clones 0, 1, 2: at least 90 % of each one's graph cells under one clone number, three numbers
    cells = np.arange(96)
    numbers = []
    for q in range(3):
        lab = want[(cells % 4 == q) & (want > 0)]
        top = np.bincount(lab).argmax()
        assert (lab == top).mean() >= 0.9, (q, np.bincount(lab))
        numbers.append(top)
    assert len(set(numbers)) == 3
    table = clone_variants(res, got, engine)
    assert len(table) == got.n_clones * len(called)
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------- pipeline
@pytest.mark.parametrize("fmt", ["standard", "hdf5"])
def test_pipeline_find_clones(engine, planted, tmp_path, fmt):
    from mgatk2_b200 import BAMReader, PipelineConfig, run_pipeline
    from mgatk2_b200.bamio import write_bam
    from mgatk2_b200.barcodes import load_barcodes
    from mgatk2_b200.clones import clone_variants, find_clones, read_clone_variants, read_clones
    from mgatk2_b200.synth import make_whitelist
    batch, _, _, _ = planted
    barcodes = make_whitelist(96, seed=3)
    bam = str(tmp_path / "possorted_bam.bam")
    write_bam(bam, batch, barcodes, ref_lens=(248956422, P_SHORT, 156040895), write_index=False)
    kw = dict(barcode_file=None, min_barcode_reads=10, output_format=fmt, mito_length=P_SHORT, max_strand_bias=1.0)
    run_pipeline(bam, str(tmp_path / "plain"), **kw)
    run_pipeline(bam, str(tmp_path / "clones"), find_clones=True, **kw)
    plain, got = _files(tmp_path / "plain"), _files(tmp_path / "clones")
    extra = {"output/variant_stats.tsv.gz", "output/variant_cells.tsv.gz", "output/clones.tsv.gz",
             "output/clone_variants.tsv.gz"}
    assert set(got) == set(plain) | extra
    for k in plain:
        if k == "qc/summary.txt":
            assert _summary_body(plain[k]) == _summary_body(got[k])
        else:
            assert plain[k] == got[k], k
    run_pipeline(bam, str(tmp_path / "called"), call_variants=True, **kw)
    called_files = _files(tmp_path / "called")
    for k in ("output/variant_stats.tsv.gz", "output/variant_cells.tsv.gz"):
        assert called_files[k] == got[k], k
    # the files against find_clones / clone_variants of the seam's own result
    wl, _ = load_barcodes(None, bam, barcode_tag="CB", mito_chr="chrM", min_barcode_reads=10)
    cfg = PipelineConfig(mito_length=P_SHORT, max_strand_bias=1.0)
    rbb, _ = BAMReader(bam, cfg, set(wl), barcode_list=list(wl)).collect_reads_by_barcode()
    res = rbb.result
    clones = find_clones(res, engine=engine)
    cols = res.columns if res.columns is not None else np.arange(len(res.planes))
    names, labels = read_clones(os.path.join(tmp_path, "clones", "output", "clones.tsv.gz"))
    sel = np.nonzero(clones.selected)[0]
    assert names == [wl[int(cols[k])] for k in sel]
    np.testing.assert_array_equal(labels, clones.labels[sel])
    assert clones.n_clones >= 3
    table = clone_variants(res, clones, engine)
    back = read_clone_variants(os.path.join(tmp_path, "clones", "output", "clone_variants.tsv.gz"))
    for f in ("clone", "variant", "n_cells", "n_cells_detected"):
        np.testing.assert_array_equal(back[f], table[f], err_msg=f)
    np.testing.assert_allclose(back["mean_heteroplasmy"], table["mean_heteroplasmy"], rtol=1e-9)
