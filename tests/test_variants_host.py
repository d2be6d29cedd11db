"""CPU checks of the variant statistics (mgatk2_b200/variants.py, oracle/variants.py): hand-computed answers on a few
cells and positions, the host floats against a direct dense computation, the dtype against the C struct and the two
files read back."""
import ctypes
import gzip
import math

import numpy as np
import pytest

from mgatk2_b200.exceptions import ProcessingError
from mgatk2_b200.variants import (VARIANT_SUMS_DTYPE, call_variants, finalize, read_variant_stats, write_variant_cells,
                                  write_variant_stats)
from oracle.variants import oracle_variant_sums, reference_alleles

A, C, G, T = range(4)


def cells(spec, P=1, ref_letter=A, extra_ref=50):
    """counts [n, P, 4, 2] / coverage [n, P] from per-cell (f, r) of letter C at position 0; the reference letter gets
    `extra_ref` forward reads so that coverage = a + extra_ref."""
    n = len(spec)
    counts = np.zeros((n, P, 4, 2), np.uint32)
    for i, (f, r) in enumerate(spec):
        counts[i, 0, C] = (f, r)
        counts[i, 0, ref_letter, 0] = extra_ref
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    return counts, cov


def row(table, name):
    hit = table[table["variant"] == name]
    assert len(hit) == 1, name
    return hit[0]


def test_dtype_matches_the_c_struct():
    from mgatk2_b200._lib import VariantSumsC
    assert VARIANT_SUMS_DTYPE.itemsize == ctypes.sizeof(VariantSumsC) == 128
    for name, *_ in VariantSumsC._fields_:
        assert VARIANT_SUMS_DTYPE.fields[name][1] == getattr(VariantSumsC, name).offset, name


def test_strand_correlation_known_value():
    counts, cov = cells([(1, 2), (2, 4), (3, 7)])
    s = oracle_variant_sums(counts, cov, np.array([A]))
    t = finalize(s, 3)
    r = row(t, "1A>C")
    # n = 3, sums 6, 13, 14, 69, 31: (3*31 - 6*13) / sqrt((3*14 - 36) * (3*69 - 169)) = 15 / sqrt(228)
    assert r["strand_correlation"] == 15 / math.sqrt(228)
    assert (s[0, C]["sum_ff"], s[0, C]["sum_rr"], s[0, C]["sum_fr"]) == (14, 69, 31)
    assert row(t, "1A>G")["n_cells_detected"] == 0 and math.isnan(row(t, "1A>G")["strand_correlation"])


def test_strand_correlation_nan():
    counts, cov = cells([(3, 4), (0, 0), (0, 0)])            # one cell with a > 0
    assert math.isnan(row(finalize(oracle_variant_sums(counts, cov, np.array([A])), 3), "1A>C")["strand_correlation"])
    counts, cov = cells([(2, 1), (2, 3), (2, 5)])            # forward strand constant
    t = finalize(oracle_variant_sums(counts, cov, np.array([A])), 3)
    assert math.isnan(row(t, "1A>C")["strand_correlation"])


def test_variance_stabilised_below_low_coverage():
    # (a, d) = (10, 20), (1, 5), (2, 10); L = 10: the middle cell is set to the mean 13 / 35
    counts, cov = cells([(10, 0), (1, 0), (2, 0)], extra_ref=0)
    counts[:, 0, A, 0] = np.array([20, 5, 10]) - np.array([10, 1, 2])
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    s = oracle_variant_sums(counts, cov, np.array([A]), low_coverage_threshold=10)
    r = row(finalize(s, 3), "1A>C")
    mean = 13 / 35
    assert r["mean"] == mean
    want = np.var([0.5, mean, 0.2], ddof=1)
    assert r["variance"] == pytest.approx(want, rel=1e-12)
    assert r["vmr"] == pytest.approx(want / (mean + 1e-11), rel=1e-12)
    assert r["n_cells_low_coverage"] == 1 and s[0, C]["n_low"] == 1


def test_thresholds_exactly_at_the_fraction():
    a = [4, 5, 9, 10, 19, 20, 94, 95]                         # d = 100
    counts, cov = cells([(x, 0) for x in a], extra_ref=0)
    counts[:, 0, A, 0] = 100 - np.array(a)
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    r = row(finalize(oracle_variant_sums(counts, cov, np.array([A])), len(a)), "1A>C")
    assert [r[f"n_cells_over_{k}"] for k in (5, 10, 20, 95)] == [7, 5, 3, 1]
    a = [1, 2, 4, 19]                                         # d = 20: exactly 5 %, 10 %, 20 %, 95 %
    counts, cov = cells([(x, 0) for x in a], extra_ref=0)
    counts[:, 0, A, 0] = 20 - np.array(a)
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    r = row(finalize(oracle_variant_sums(counts, cov, np.array([A])), len(a)), "1A>C")
    assert [r[f"n_cells_over_{k}"] for k in (5, 10, 20, 95)] == [4, 3, 2, 1]


def test_max_heteroplasmy_tie_keeps_the_first_cell():
    for spec, want in (([(1, 0), (2, 0), (3, 0), (1, 0)], (1, 4)), ([(2, 0), (1, 0)], (2, 8))):
        counts, cov = cells(spec, extra_ref=0)
        d = {1: 4, 2: 8, 3: 12} if want == (1, 4) else {2: 8, 1: 4}
        dd = np.array([d[f] for f, _ in spec])
        if want == (1, 4):
            dd[-1] = 5                                        # 1 / 5 is below the tie
        counts[:, 0, A, 0] = dd - np.array([f for f, _ in spec])
        cov = counts.sum(axis=(2, 3)).astype(np.uint32)
        s = oracle_variant_sums(counts, cov, np.array([A]))
        assert (int(s[0, C]["max_alt"]), int(s[0, C]["max_cov"])) == want
        assert row(finalize(s, len(spec)), "1A>C")["max_heteroplasmy"] == want[0] / want[1]


def test_reference_n_positions_give_no_variant():
    counts, cov = cells([(3, 3), (2, 2)], P=3)
    bt = np.zeros((3, 4), np.int64)
    bt[0, A], bt[2, G] = 100, 7
    bt[2, T] = 7                                              # tie: the first letter wins
    ref = reference_alleles(bt)
    assert ref.tolist() == [A, -1, G]
    s = oracle_variant_sums(counts, cov, ref)
    assert not s[1]["valid"].any() and s[0]["valid"].tolist() == [0, 1, 1, 1] and s[2]["valid"].tolist() == [1, 1, 0, 1]
    t = finalize(s, 2)
    assert sorted(set(t["position"].tolist())) == [1, 3]
    assert t["variant"].tolist()[:3] == ["1A>C", "1A>G", "1A>T"] and t["nucleotide"].tolist()[3:] == ["G>A", "G>C", "G>T"]


def test_masked_out_cells():
    rng = np.random.default_rng(3)
    counts = rng.integers(0, 6, size=(5, 3, 4, 2)).astype(np.uint32)
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    ref = np.array([A, C, T])
    mask = np.array([True, False, True, True, False])
    got = oracle_variant_sums(counts, cov, ref, mask)
    want = oracle_variant_sums(counts[mask], cov[mask], ref)
    assert got.tobytes() == want.tobytes()
    assert finalize(got, 3).tobytes() == finalize(want, 3).tobytes()


def test_zero_and_one_cell():
    counts, cov = cells([(3, 4)])
    t0 = finalize(oracle_variant_sums(counts, cov, np.array([A]), np.array([False])), 0)
    r = row(t0, "1A>C")
    assert r["n_cells_covered"] == 0 and r["mean"] == 0 and math.isnan(r["variance"]) and math.isnan(r["mean_coverage"])
    assert math.isnan(r["max_heteroplasmy"]) and math.isnan(r["strand_correlation"])
    t1 = finalize(oracle_variant_sums(counts, cov, np.array([A])), 1)
    r = row(t1, "1A>C")
    assert r["mean"] == 7 / 57 and r["mean_coverage"] == 57 and math.isnan(r["variance"])
    assert r["max_heteroplasmy"] == 7 / 57 and r["n_cells_conf_detected"] == 1


def test_finalize_against_a_dense_computation():
    rng = np.random.default_rng(11)
    Cn, P, L = 40, 30, 10
    counts = rng.integers(0, 9, size=(Cn, P, 4, 2)).astype(np.uint32)
    counts[rng.random((Cn, P, 4, 2)) < 0.4] = 0
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    bt = counts.sum(axis=(0, 3)).astype(np.int64)
    ref = reference_alleles(bt)
    mask = rng.random(Cn) < 0.8
    t = finalize(oracle_variant_sums(counts, cov, ref, mask, L), int(mask.sum()))
    cc, dd = counts[mask].astype(np.float64), cov[mask].astype(np.float64)
    for r in t:
        p, b = int(r["position"]) - 1, "ACGT".index(r["alt"])
        f, rv, d = cc[:, p, b, 0], cc[:, p, b, 1], dd[:, p]
        a = f + rv
        mean = a.sum() / d.sum() if d.sum() else 0.0
        assert r["mean"] == mean
        with np.errstate(divide="ignore", invalid="ignore"):
            het = np.where(d >= L, a / d, mean)
        assert r["variance"] == pytest.approx(np.var(het, ddof=1), rel=1e-9, abs=1e-15)
        det = a > 0
        if det.sum() >= 2 and f[det].std() > 0 and rv[det].std() > 0:
            assert r["strand_correlation"] == pytest.approx(np.corrcoef(f[det], rv[det])[0, 1], rel=1e-12)
        else:
            assert math.isnan(r["strand_correlation"])
        assert r["n_cells_conf_detected"] == int(((f >= 2) & (rv >= 2)).sum())
        cover = d > 0
        assert r["max_heteroplasmy"] == ((a[cover] / d[cover]).max() if cover.any() else r["max_heteroplasmy"])


def test_sum_cov_limit():
    s = np.zeros((1, 4), VARIANT_SUMS_DTYPE)
    s["sum_cov"] = 1 << 32
    with pytest.raises(ProcessingError):
        finalize(s, 1)


def test_call_variants_filter():
    t = np.zeros(4, finalize(np.zeros((0, 4), VARIANT_SUMS_DTYPE), 0).dtype)
    t["n_cells_conf_detected"] = [5, 4, 5, 5]
    t["strand_correlation"] = [0.65, 0.9, np.nan, 0.9]
    t["vmr"] = [0.0100001, 1.0, 1.0, 0.01]
    assert call_variants(t).tolist() == t[:1].tolist()
    assert len(call_variants(t, min_conf_detected=4, min_vmr=0.0)) == 3


def test_files_round_trip(tmp_path):
    rng = np.random.default_rng(5)
    counts = rng.integers(0, 9, size=(6, 4, 4, 2)).astype(np.uint32)
    cov = counts.sum(axis=(2, 3)).astype(np.uint32)
    cov[2, 1] = 0
    counts[2, 1] = 0
    ref = np.array([A, -1, G, T])
    t = finalize(oracle_variant_sums(counts, cov, ref), 6)
    write_variant_stats(t, tmp_path / "variant_stats.tsv.gz")
    back = read_variant_stats(tmp_path / "variant_stats.tsv.gz")
    assert back.dtype == t.dtype and len(back) == len(t)
    for name in t.dtype.names:
        if t.dtype[name].kind == "f":
            np.testing.assert_allclose(back[name], t[name], rtol=1e-9, equal_nan=True)
        else:
            assert back[name].tolist() == t[name].tolist(), name
    text = gzip.open(tmp_path / "variant_stats.tsv.gz", "rt").read().splitlines()
    assert text[0].split("\t")[:3] == ["variant", "position", "nucleotide"] and len(text) == len(t) + 1
    called = t[:2]
    ids = (called["position"] - 1) * 4 + np.array(["ACGT".index(x) for x in called["alt"]])
    per_cell = np.stack([np.stack([counts[:, i // 4, i % 4, 0], counts[:, i // 4, i % 4, 1], cov[:, i // 4]]) for i in ids])
    mask = np.array([True, True, True, False, True, True])
    names = [f"BC{k}-1" for k in range(6)]
    write_variant_cells(called, per_cell, names, mask, tmp_path / "variant_cells.tsv.gz")
    lines = gzip.open(tmp_path / "variant_cells.tsv.gz", "rt").read().splitlines()
    assert lines[0] == "variant\tbarcode\talt_fwd\talt_rev\tcoverage"
    want = [f"{called['variant'][i]}\t{names[k]}\t{per_cell[i, 0, k]}\t{per_cell[i, 1, k]}\t{per_cell[i, 2, k]}"
            for i in range(len(called)) for k in range(6) if mask[k] and per_cell[i, 2, k] > 0]
    assert lines[1:] == want
