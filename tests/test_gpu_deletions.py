"""GPU checks of the deletion scan (mgatk_deletion_scan_device, mgatk2_b200/deletions.py) against the plain-Python
restatement in oracle/deletions.py.

1. Planted batches (synth_deletions) at 2x50 and 2x150 bp, with and without D-gap reads, in all three dedup modes:
   counts and all four histograms equal the oracle exactly, on outputs pre-filled with a nonzero pattern (the entry adds).
2. Contig lengths 1 000, 16 569 and 70 000; 20 000 barcode columns drawn from skewed weights; a run of 100 000
   duplicates starting on a breakpoint behind a first copy that is not relevant.
3. Three parts cut on start borders add up to the one-batch answer.
4. Status codes of bad arguments, unsorted records, reads beyond max_read_extent and deletions out of range; destroying
   a handle frees its scratch.
5. find_deletions on the GPU histograms recovers every planted deletion; the pipeline with `deletions` and
   `find_deletions` adds two files and leaves every other file byte-identical, one batch and streamed.
"""
import ctypes
import gzip

import numpy as np
import pytest

from oracle import deletions as od

pytestmark = pytest.mark.gpu

K = 16
PLANTED = ((8470, 13446), (6330, 13994), (1500, 2100))


@pytest.fixture(scope="module")
def engine():
    from mgatk2_b200.pileup import get_engine
    return get_engine(0)


def lr_of(dels):
    return [(f - 2, t) for f, t in dels]


def device_scan(engine, batch, n_cells, P, dels, dedup_mode=0, min_mapq=30, min_clip=5, find=True, extent=None):
    """One call on outputs pre-filled with a pattern; returns (counts, end_clip, start_clip, end_seq, start_seq, error
    bits) with the pattern taken off again."""
    import torch
    from mgatk2_b200.config import PipelineConfig
    dev = torch.device("cuda", engine.device)
    cfg = PipelineConfig(mito_length=P, min_mapq=min_mapq, skip_deduplication=dedup_mode == 2,
                         use_fragment_length_dedup=dedup_mode == 0)
    assert cfg.dedup.mode == dedup_mode
    params = cfg.to_params(n_cells, extent or max(batch.max_read_extent(), 1))
    lr = np.array(lr_of(dels), np.int32).reshape(-1, 2)
    D = len(lr)
    pat_c = (np.arange(max(D * 4 * n_cells, 1), dtype=np.int64) * 7 % 13 + 1).astype(np.uint32)
    pat_h = (np.arange(2 * P, dtype=np.int64) * 5 % 11 + 3).astype(np.uint64)
    pat_s = (np.arange(2 * P * K * 4, dtype=np.int64) % 17 + 1).astype(np.uint64)
    counts = torch.from_numpy(pat_c.view(np.int32).copy()).to(dev)
    hist = torch.from_numpy(pat_h.view(np.int64).copy()).to(dev)
    seq = torch.from_numpy(pat_s.view(np.int64).copy()).to(dev)
    err = torch.zeros(1, dtype=torch.int64, device=dev)
    ends = torch.from_numpy(np.ascontiguousarray(lr.T.reshape(-1))).to(dev)
    db = engine.upload(batch)
    bc = db.as_c()
    stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    rc = engine.lib.mgatk_deletion_scan_device(engine.handle, ctypes.byref(params), ctypes.byref(bc), min_clip,
                                               ends.data_ptr(), ends.data_ptr() + 4 * D, D, counts.data_ptr(),
                                               hist.data_ptr() if find else None, seq.data_ptr() if find else None,
                                               err.data_ptr(), stream)
    assert rc == 0, engine.lib.mgatk_last_error(engine.handle)
    torch.cuda.synchronize(dev)
    c = (counts.cpu().numpy().view(np.uint32) - pat_c)[: D * 4 * n_cells].reshape(D, 4, n_cells)
    h = (hist.cpu().numpy().view(np.uint64) - pat_h).reshape(2, P)
    s = (seq.cpu().numpy().view(np.uint64) - pat_s).reshape(2, P, K, 4)
    if not find:
        assert not h.any() and not s.any()
    return c, h[0], h[1], s[0], s[1], int(err.cpu()[0])


def assert_equals_oracle(engine, batch, n_cells, P, dels, dedup_mode=0, min_mapq=30, find=True):
    c, ec, sc, es, ss, err = device_scan(engine, batch, n_cells, P, dels, dedup_mode, min_mapq, find=find)
    assert err == 0
    o = od.scan(batch, n_cells, P, lr_of(dels), dedup_mode=dedup_mode, min_mapq=min_mapq, find=find)
    np.testing.assert_array_equal(c, o["counts"])
    if find:
        np.testing.assert_array_equal(ec, o["end_clip"])
        np.testing.assert_array_equal(sc, o["start_clip"])
        np.testing.assert_array_equal(es, o["end_seq"])
        np.testing.assert_array_equal(ss, o["start_seq"])
    return o


@pytest.mark.parametrize("read_len,gap_reads", [(50, False), (50, True), (150, True)])
@pytest.mark.parametrize("dedup_mode", [0, 1, 2])
def test_planted_equals_oracle(engine, read_len, gap_reads, dedup_mode):
    from mgatk2_b200.synth import synth_deletions
    batch, _, _ = synth_deletions(read_len=read_len, gap_reads=gap_reads, seed=100 + read_len)
    o = assert_equals_oracle(engine, batch, 40, 16569, PLANTED, dedup_mode=dedup_mode)
    assert o["counts"][:, :2].sum() > 100 and o["counts"][:, 3].sum() > 100
    assert o["counts"][:, 2].sum() == (len(PLANTED) if gap_reads else 0)
    # without discovery the CIGAR is read near the breakpoints only: the counts stay the same
    assert_equals_oracle(engine, batch, 40, 16569, PLANTED, dedup_mode=dedup_mode, find=False)


@pytest.mark.parametrize("P,dels", [(1000, ((302, 700), (120, 260))), (16569, PLANTED),
                                    (70000, ((8470, 13446), (40000, 61000)))])
def test_contig_lengths(engine, P, dels):
    from mgatk2_b200.synth import synth_deletions
    batch, _, _ = synth_deletions(n_cells=25, n_fragments=4000, deletions=dels, mito_length=P, read_len=75, seed=P,
                                  n_background=2000)
    assert_equals_oracle(engine, batch, 25, P, dels)


def test_skewed_columns(engine):
    from mgatk2_b200.synth import synth_deletions
    batch, _, _ = synth_deletions(n_cells=20000, n_fragments=30000, read_len=150, skew=2.0, seed=9, n_background=5000)
    assert_equals_oracle(engine, batch, 20000, 16569, PLANTED)


def test_hot_spot_duplicates_on_a_breakpoint(engine):
    from mgatk2_b200.batch import ReadBatch
    from mgatk2_b200.synth import synth_deletions
    batch, ref, _ = synth_deletions(n_cells=20, n_fragments=3000, seed=5)
    l, r = PLANTED[0][0] - 2, PLANTED[0][1]
    first = {"pos": r, "cigar": [(0, 50)], "seq": ref[r: r + 50], "bc_idx": 3, "flag": 99, "mapq": 60, "tlen": 250}
    clip = dict(first, cigar=[(4, 20), (0, 30)], seq=ref[l - 19: l + 1] + ref[r: r + 30])
    other = dict(clip, bc_idx=4)                              # another cell: its first copy survives
    dups = ReadBatch.from_records([first] + [clip] * 100000 + [other] * 5)
    both = ReadBatch.concat([batch, dups])
    both = both.take(np.argsort(both.pos, kind="stable"))
    o = assert_equals_oracle(engine, both, 20, 16569, PLANTED)
    base = od.scan(batch, 20, 16569, lr_of(PLANTED), find=True)
    assert o["counts"][0, 1, 3] == base["counts"][0, 1, 3] and o["counts"][0, 1, 4] == base["counts"][0, 1, 4] + 1
    c, *_ = device_scan(engine, both, 20, 16569, PLANTED, dedup_mode=2)
    assert c[0, 1, 3] == base["counts"][0, 1, 3] + 100000


def test_parts_add_up(engine):
    from mgatk2_b200.config import PipelineConfig
    from mgatk2_b200.deletions import scan_deletions
    from mgatk2_b200.synth import synth_deletions
    batch, _, _ = synth_deletions(read_len=150, seed=31)
    cfg = PipelineConfig()
    one = scan_deletions(batch, cfg, 40, deletions=PLANTED, find=True)
    parts = batch.split_on_start_borders(3)
    assert len(parts) == 3
    three = scan_deletions(iter(parts), cfg, 40, deletions=PLANTED, find=True)
    for k in ("counts", "end_clip", "start_clip", "end_seq", "start_seq"):
        np.testing.assert_array_equal(getattr(one, k), getattr(three, k))
    o = od.scan(batch, 40, 16569, lr_of(PLANTED), find=True)
    np.testing.assert_array_equal(one.counts, o["counts"])


def test_status_codes(engine):
    import torch
    from mgatk2_b200.config import PipelineConfig
    from mgatk2_b200.deletions import scan_deletions
    from mgatk2_b200.exceptions import PileupKernelError
    from mgatk2_b200.synth import synth_deletions
    batch, _, _ = synth_deletions(n_cells=8, n_fragments=500, n_background=200, seed=2)
    lib, h = engine.lib, engine.handle
    dev = torch.device("cuda", 0)
    cfg = PipelineConfig()
    params = cfg.to_params(8, batch.max_read_extent())
    db = engine.upload(batch)
    bc = db.as_c()
    ends = torch.tensor([100, 300, 900, 20000], dtype=torch.int32, device=dev)     # l = 100, 300; r = 900, 20000
    out = torch.zeros(4 * 4 * 8, dtype=torch.int32, device=dev)
    hist = torch.zeros(2 * 16569, dtype=torch.int64, device=dev)
    seq = torch.zeros(2 * 16569 * K * 4, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int64, device=dev)
    s = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    e, o, hp, sp = err.data_ptr(), out.data_ptr(), hist.data_ptr(), seq.data_ptr()
    l0, r0 = ends.data_ptr(), ends.data_ptr() + 8

    def call(p=params, b=bc, mc=5, left=l0, right=r0, n=1, c=o, hh=hp, ss=sp, ee=e):
        return lib.mgatk_deletion_scan_device(h, ctypes.byref(p) if p is not None else None,
                                              ctypes.byref(b) if b is not None else None, mc, left, right, n, c, hh, ss,
                                              ee, s)
    assert call() == 0
    assert lib.mgatk_deletion_scan_device(None, ctypes.byref(params), ctypes.byref(bc), 5, l0, r0, 1, o, hp, sp, e, s) == 1
    assert call(p=None) == 1 and call(b=None) == 1 and call(ee=None) == 1
    assert call(mc=0) == 1 and call(n=-1) == 1 and call(left=None) == 1 and call(c=None) == 1
    assert call(hh=None) == 1 and call(ss=None) == 1
    assert call(hh=None, ss=None) == 0                       # no discovery
    assert call(n=1025) == 8
    bad = cfg.to_params(8, batch.max_read_extent())
    bad.dedup_mode = 3
    assert call(p=bad) == 1
    bad = cfg.to_params(8, 0)
    assert call(p=bad) == 1
    bad = cfg.to_params(8, (1 << 20) + 1)
    assert call(p=bad) == 5
    bad = cfg.to_params(8, batch.max_read_extent())
    bad.mito_length = 1 << 24
    assert call(p=bad) == 8
    torch.cuda.synchronize(dev)
    assert int(err.cpu()[0]) == 0
    assert call(n=2) == 0                                     # (300, 20000): r beyond P -> error bit 16
    torch.cuda.synchronize(dev)
    assert int(err.cpu()[0]) == 16
    st = np.zeros(8, np.uint64)
    st[7] = 16
    assert lib.mgatk_check_stats(st.ctypes.data) == 8
    with pytest.raises(ValueError):
        scan_deletions(batch, cfg, 8, deletions=[(10, 20000)])                    # r beyond the contig
    unsorted = batch.take(np.r_[np.arange(1, batch.n_records), 0])
    with pytest.raises(PileupKernelError) as ex:
        scan_deletions(unsorted, cfg, 8, deletions=PLANTED)
    assert ex.value.args[0] == 4 or "sorted" in str(ex.value)
    _, _, _, _, _, bits = device_scan(engine, batch, 8, 16569, PLANTED, find=True, extent=60)   # the gap reads are longer
    assert bits & 2


def test_destroy_frees_scratch():
    import torch
    from mgatk2_b200.engine import PileupEngine
    from mgatk2_b200.synth import synth_batch
    batch = synth_batch(200, 2_000_000, "atac50", seed=3)
    eng = PileupEngine(0)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free0 = torch.cuda.mem_get_info(0)[0]
    device_scan(eng, batch, 200, 16569, PLANTED)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    free1 = torch.cuda.mem_get_info(0)[0]
    scratch = 2_000_000 * 4 + (1 << 22) * 16                    # relevant list + dedup table: about 72 MB
    assert free0 - free1 >= scratch
    eng.close()
    free2 = torch.cuda.mem_get_info(0)[0]
    assert free2 - free1 >= scratch


def test_find_recovers_planted(engine):
    from mgatk2_b200.config import PipelineConfig
    from mgatk2_b200.deletions import deletion_heteroplasmy, find_deletions, scan_deletions
    from mgatk2_b200.synth import synth_deletions
    for read_len in (50, 150):
        batch, ref, het = synth_deletions(read_len=read_len, seed=77 + read_len)
        scan = scan_deletions(batch, PipelineConfig(), 40, find=True)
        cands = find_deletions(scan, ref)
        assert sorted((int(c["first"]), int(c["last"])) for c in cands) == sorted(PLANTED)
        assert set(cands["support"].tolist()) == {"both"}
        counted = scan_deletions(batch, PipelineConfig(), 40, deletions=cands)
        t = deletion_heteroplasmy(counted)
        for row in t[~np.isnan(t["heteroplasmy"])]:
            want = het[row["cell"], [f"m.{f}_{l}del" for f, l in PLANTED].index(row["deletion"])]
            if row["clip_left"] + row["clip_right"] + row["gap"] + row["wt"] >= 30:
                assert abs(row["heteroplasmy"] - want) < 0.35


@pytest.mark.parametrize("streamed", [False, True])
def test_pipeline(engine, tmp_path, streamed):
    from mgatk2_b200 import run_pipeline
    from mgatk2_b200.bamio import write_bam
    from mgatk2_b200.deletions import read_deletion_candidates, read_deletions
    from mgatk2_b200.synth import make_whitelist, synth_deletions
    from tests.test_gpu_variants import _files, _summary_body
    batch, _, _ = synth_deletions(read_len=75, seed=12)
    barcodes = make_whitelist(40, seed=4)
    bam = str(tmp_path / "possorted_bam.bam")
    write_bam(bam, batch, barcodes, write_index=False)
    kw = dict(barcode_file=None, min_barcode_reads=10, max_batch_records=4000 if streamed else None)
    run_pipeline(bam, str(tmp_path / "base"), **kw)
    run_pipeline(bam, str(tmp_path / "del"), deletions=[PLANTED[0]], find_deletions=True, **kw)
    base, got = _files(tmp_path / "base"), _files(tmp_path / "del")
    assert set(got) == set(base) | {"output/deletions.tsv.gz", "output/deletion_candidates.tsv.gz"}
    for k in base:
        if k == "qc/summary.txt":
            assert _summary_body(base[k]) == _summary_body(got[k])
        else:
            assert base[k] == got[k], k
    cands = read_deletion_candidates(tmp_path / "del" / "output" / "deletion_candidates.tsv.gz")
    assert sorted((int(c["first"]), int(c["last"])) for c in cands) == sorted(PLANTED)
    rows = read_deletions(tmp_path / "del" / "output" / "deletions.tsv.gz")
    o = od.scan(batch, 40, 16569, lr_of(PLANTED))["counts"]
    names = [f"m.{f}_{l}del" for f, l in PLANTED]
    assert {r["deletion"] for r in rows} == set(names)
    for r in rows:
        c = o[names.index(r["deletion"]), :, barcodes.index(r["barcode"])]
        assert [r["clip_left"], r["clip_right"], r["gap"], r["wt"]] == c.tolist()
        d = int(c[:3].sum())
        assert r["heteroplasmy"] == float(format(d / (d + int(c[3])), ".10g"))       # written '.10g'
    n_rows = sum(1 for d in range(3) for c in range(40) if o[d, :, c].sum() > 0)
    assert len(rows) <= n_rows and len(rows) >= n_rows - 3 * 3            # a few cells may fail the QC gate
    assert gzip.open(tmp_path / "del" / "output" / "deletions.tsv.gz", "rt").readline().startswith("barcode\tdeletion\t")
