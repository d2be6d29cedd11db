"""Host checks of the clone markers (DESIGN §8 "Clone markers"): the host formula of markers.py against scipy's
asymptotic Mann-Whitney U test with continuity correction, a hand-computed case, oracle/markers.py against
scipy.stats.rankdata, the Bonferroni cap, the table layout and `clone_markers.tsv.gz` round-tripping."""
import math

import numpy as np
import pytest
import scipy.stats as ss

from mgatk2_b200.markers import (CLONE_MARKERS_DTYPE, MARKERS_DTYPE, bonferroni, read_clone_markers, wilcoxon,
                                 write_clone_markers)
from oracle import markers as om


def exact_ranks(group, rest):
    """(rank2 of `group`, ties) of the values of group + rest by the oracle."""
    r2, ties = om.mid_ranks2(np.concatenate([group, rest]))
    return int(r2[: len(group)].sum()), ties


def seeded_cases():
    rng = np.random.default_rng(11)
    cases = []
    for n1, n2, zero in [(30, 70, 0.9), (5, 400, 0.97), (200, 300, 0.5), (12, 13, 0.0), (1, 50, 0.6), (1, 1, 0.0)]:
        g = np.where(rng.random(n1) < zero, 0.0, rng.integers(1, 6, n1) / rng.integers(1, 8, n1))
        r = np.where(rng.random(n2) < zero, 0.0, rng.integers(1, 6, n2) / rng.integers(1, 8, n2))
        cases.append((g, r))
    cases.append((np.linspace(0.5, 1.0, 200), np.linspace(0.0, 0.4, 200)))     # very small p
    cases.append((np.array([1.0, 4.0]), np.array([2.0, 3.0])))                 # U = mu
    cases.append((np.array([0.5]), np.array([0.5, 0.0, 0.25])))                # one member with a tie
    return cases


@pytest.mark.parametrize("k", range(len(seeded_cases())))
def test_formula_against_scipy(k):
    g, r = seeded_cases()[k]
    rank2, ties = exact_ranks(g, r)
    U, auc, z, p = wilcoxon(rank2, ties, len(g), len(g) + len(r))
    want = ss.mannwhitneyu(g, r, alternative="two-sided", method="asymptotic", use_continuity=True)
    assert U == want.statistic
    np.testing.assert_allclose(p, want.pvalue, rtol=1e-9)
    assert auc == U / (len(g) * len(r))
    if k == len(seeded_cases()) - 3:
        assert p < 1e-60
    if k == len(seeded_cases()) - 2:
        assert U == 2 and z == 0 and p == 1.0


def test_all_tied_and_empty_sides_are_nan():
    rank2, ties = exact_ranks(np.full(4, 0.25), np.full(6, 0.25))
    assert ties == 10 ** 3 - 10
    U, auc, z, p = wilcoxon(rank2, ties, 4, 10)
    assert U == 12 and math.isnan(auc) and math.isnan(z) and math.isnan(p)
    assert math.isnan(ss.mannwhitneyu(np.full(4, 0.25), np.full(6, 0.25), method="asymptotic").pvalue)
    for n1, N in [(0, 5), (5, 5)]:                                             # n1 = 0, n2 = 0
        rank2 = n1 * (N + 1)
        assert all(math.isnan(v) for v in wilcoxon(rank2, N ** 3 - N, n1, N)[1:])


def test_hand_computed():
    """In-group x = [0.5, 0], rest [0, 0, 0.25]: ranks 0 0 0 -> 2, 0.25 -> 4, 0.5 -> 5, so rank2 = 2 (5 + 2), and the run
    of three zeros gives ties = 27 - 3."""
    rank2, ties = exact_ranks(np.array([0.5, 0.0]), np.array([0.0, 0.0, 0.25]))
    assert (rank2, ties) == (14, 24)
    U, auc, z, p = wilcoxon(14, 24, 2, 5)
    assert U == 4.0 and auc == 4 / 6                                           # 7 - 3
    var = 6 / 12 * (6 - 24 / 20)
    assert z == (1 - 0.5) / math.sqrt(var) and p == math.erfc(abs(z) / math.sqrt(2))


def test_oracle_against_rankdata():
    rng = np.random.default_rng(3)
    counts = rng.integers(0, 5, (6, 3, 400)).astype(np.uint32)
    counts[:, 2] = rng.integers(0, 9, (6, 400))
    counts[:, 0, rng.random(400) < 0.5] = 0
    labels = rng.integers(-1, 6, 400)
    G = 4                                                                       # labels 5 and -1, 0: not in the test
    rank2, ties = om.marker_ranks(counts, labels, G)
    from oracle.clones import allele_frequencies
    x = allele_frequencies(counts)
    inside = (labels >= 1) & (labels <= G)
    for v in range(6):
        r = ss.rankdata(x[v, inside])
        for g in range(1, G + 1):
            assert rank2[v, g - 1] == round(2 * r[labels[inside] == g].sum())
        _, t = np.unique(x[v, inside], return_counts=True)
        assert ties[v] == int((t.astype(np.int64) ** 3 - t).sum())
    assert rank2.dtype == np.uint64 and ties.dtype == np.uint64


def test_bonferroni_cap():
    p = np.array([0.001, 0.2, 0.5, math.nan, 1.0, 0.0])
    got = bonferroni(p, 4)
    np.testing.assert_array_equal(got[[0, 1, 4, 5]], [0.004, 0.8, 1.0, 0.0])
    assert got[2] == 1.0 and math.isnan(got[3])


def test_dtype_column_order():
    rest = ["variant", "n_cells", "n_cells_rest", "n_cells_detected", "n_cells_detected_rest", "mean_heteroplasmy",
            "mean_heteroplasmy_rest", "auc", "statistic", "p_value", "p_value_adj"]
    assert list(MARKERS_DTYPE.names) == ["group", *rest]
    assert list(CLONE_MARKERS_DTYPE.names) == ["clone", *rest]


def test_file_round_trip(tmp_path):
    t = np.zeros(4, CLONE_MARKERS_DTYPE)
    t["clone"] = [1, 1, 2, 2]
    t["variant"] = ["302A>G", "16519T>C", "302A>G", "16519T>C"]
    t["n_cells"] = [10, 10, 0, 0]
    t["n_cells_rest"] = [7, 7, 17, 17]
    t["n_cells_detected"] = [3, 9, 0, 0]
    t["mean_heteroplasmy"] = [0.125, 1 / 3, math.nan, math.nan]
    t["mean_heteroplasmy_rest"] = [0.0, 0.25, 0.1, 0.2]
    t["auc"] = [0.5, 0.9785714286, math.nan, math.nan]
    t["statistic"] = [35.0, 1099511627775.5, 0.0, 0.0]                         # exact beyond ten digits, half-integer
    t["p_value"] = [1.0, 3.5e-200, math.nan, math.nan]
    t["p_value_adj"] = bonferroni(t["p_value"], 2)
    path = tmp_path / "clone_markers.tsv.gz"
    write_clone_markers(t, path)
    back = read_clone_markers(path)
    assert back.dtype == CLONE_MARKERS_DTYPE
    for f in t.dtype.names:
        if t.dtype[f].kind == "f":
            np.testing.assert_allclose(back[f], t[f], rtol=1e-9, equal_nan=True, err_msg=f)
        else:
            np.testing.assert_array_equal(back[f], t[f], err_msg=f)
    assert back["statistic"].tolist() == t["statistic"].tolist()
    import gzip
    lines = gzip.open(path, "rt").read().splitlines()
    assert lines[0] == "\t".join(CLONE_MARKERS_DTYPE.names)
    assert "\t1099511627775.5\t" in lines[2] and "\tNA\t" in lines[3]
    write_clone_markers(np.zeros(0, CLONE_MARKERS_DTYPE), path)
    assert gzip.open(path, "rt").read() == lines[0] + "\n" and len(read_clone_markers(path)) == 0
