"""Host checks of the clone step (DESIGN §8 "Clones"): the numpy oracle on hand-computed cases, the library's
mgatk_louvain_host against the oracle's Louvain (no GPU needed), the SNN graph builder of clones.py against the oracle's,
and the two files round-tripping."""
import numpy as np
import pytest

from mgatk2_b200.clones import (CLONE_VARIANTS_DTYPE, CloneResult, clone_variant_table, louvain, read_clone_variants,
                                read_clones, snn_graph, write_clone_variants, write_clones)
from oracle import clones as oc


def csr_of(n, edges):
    """Symmetric CSR of undirected weighted edges {(i, j): w}, diagonal allowed."""
    a = {}
    for (i, j), w in edges.items():
        a[(i, j)] = w
        a[(j, i)] = w
    keys = sorted(a)
    indptr = np.zeros(n + 1, np.int64)
    for i, _ in keys:
        indptr[i + 1] += 1
    return np.cumsum(indptr), np.array([j for _, j in keys], np.int32), np.array([a[k] for k in keys], np.float64)


def clone_counts(n_per, V, seed, depth=20, n_clones=3, noise=0.02):
    """uint32 [V, 3, C] of cells in n_clones clones, each with its own variants at high heteroplasmy."""
    rng = np.random.default_rng(seed)
    C = n_per * n_clones
    d = rng.integers(1, depth, (V, C)).astype(np.uint32)
    het = np.where(rng.random((V, C)) < noise, rng.random((V, C)) * 0.1, 0.0)
    for c in range(n_clones):
        cols = slice(c * n_per, (c + 1) * n_per)
        for v in range(c, V, n_clones):
            het[v, cols] = rng.uniform(0.3, 0.9, n_per)
    a = np.floor(het * d).astype(np.uint32)
    f = rng.binomial(a, 0.5).astype(np.uint32)
    return np.stack([f, a - f, d], axis=1)


# ---------------------------------------------------------------------------------------------------------------- oracle
def test_allele_frequencies_and_rows():
    counts = np.zeros((2, 3, 4), np.uint32)
    counts[0, :, 0] = (1, 2, 6)          # 0.5
    counts[0, :, 1] = (0, 0, 9)          # covered, not detected
    counts[1, :, 2] = (3, 0, 0)          # no coverage: 0
    counts[1, :, 3] = (1, 1, 8)          # 0.25
    x = oc.allele_frequencies(counts)
    np.testing.assert_array_equal(x, [[0.5, 0, 0, 0], [0, 0, 0, 0.25]])
    assert oc.graph_rows(x).tolist() == [0, 3]
    assert oc.graph_rows(x, np.array([False, True, True, True])).tolist() == [3]
    assert oc.graph_rows(np.zeros((0, 4))).tolist() == []


def test_similarity_is_the_sequential_sum():
    x = np.array([[0.1, 0.2, 0.3], [0.3, 0.2, 0.1], [1e-3, 0.7, 1e-9]])
    d = oc.dots(x)
    for i in range(3):
        for j in range(3):
            acc = 0.0
            for v in range(3):
                acc = acc + x[i, v] * x[j, v]
            assert d[i, j] == acc
    nbr, sim = oc.knn(x, 3)
    inv = [1.0 / np.sqrt(d[i, i]) for i in range(3)]
    assert nbr[0].tolist() == [0, 1, 2]          # cos(0, 1) = 10/14 > cos(0, 2)
    assert sim[0, 0] == 1.0 and sim[0, 1] == (d[0, 1] * inv[0]) * inv[1]


def test_knn_ties_small_n_and_single_row():
    x = np.array([[1.0, 0.0], [0.5, 0.5], [1.0, 0.0], [2.0, 0.0], [0.0, 1.0]])
    nbr, sim = oc.knn(x, 4)
    assert nbr[0].tolist() == [0, 2, 3, 1]       # identical directions tie to the lower row
    assert nbr[3].tolist() == [3, 0, 2, 1]
    assert sim[0, 1] == sim[0, 2]
    nbr, sim = oc.knn(x[:3], 10)                 # n < k: k_eff = n
    assert nbr.shape == (3, 3) and nbr[1].tolist() == [1, 0, 2]
    nbr, sim = oc.knn(x[:1], 10)
    assert nbr.tolist() == [[0]] and sim.tolist() == [[1.0]]


def test_all_zero_row_has_cosine_zero():
    x = np.array([[1.0, 0.0], [0.0, 0.0], [0.5, 0.5]])
    nbr, sim = oc.knn(x, 3)
    assert np.isfinite(sim).all() and sim[1].tolist() == [1.0, 0.0, 0.0] and nbr[1].tolist() == [1, 0, 2]
    assert nbr[0].tolist() == [0, 2, 1] and sim[0, 2] == 0.0


def test_snn_weights_by_hand():
    nbr = np.array([[0, 1, 2], [1, 0, 2], [2, 3, 0], [3, 2, 1]], np.int32)
    w = oc.snn_weights(nbr)
    assert w[0].tolist() == [1.0, 3 / 3, 2 / 4]  # |N0 ∩ N0| = 3, |N0 ∩ N1| = 3, |N0 ∩ N2| = 2
    assert w[3].tolist() == [1.0, 2 / 4, 2 / 4]
    indptr, indices, weights = oc.snn_graph(nbr, w, prune=0.6)
    assert indptr.tolist() == [0, 2, 4, 5, 6]    # the 0.5 edges are pruned, the diagonal stays
    assert indices.tolist() == [0, 1, 0, 1, 2, 3] and weights.tolist() == [1.0] * 6
    for a, b in zip(snn_graph(nbr, w, 0.6), (indptr, indices, weights)):
        np.testing.assert_array_equal(a, b)
    assert oc.snn_graph(nbr, w)[0].tolist() == [0, 3, 7, 11, 14]    # unpruned: 0-3 is no kNN pair, 1-3 is


def test_two_triangles_and_components():
    e = {(0, 1): 1.0, (1, 2): 1.0, (0, 2): 1.0, (3, 4): 1.0, (4, 5): 1.0, (3, 5): 1.0, (2, 3): 0.1}
    labels, levels = oc.louvain(*csr_of(6, e))
    assert labels.tolist() == [1, 1, 1, 2, 2, 2] and levels >= 1
    got, _ = louvain(*csr_of(6, e))
    assert got.tolist() == labels.tolist()
    e2 = {(0, 0): 1.0, (1, 1): 1.0, (0, 1): 1.0, (2, 2): 1.0, (3, 3): 1.0, (2, 3): 1.0, (4, 4): 1.0}
    labels, _ = oc.louvain(*csr_of(5, e2))
    assert labels[0] == labels[1] and labels[2] == labels[3]
    assert len({labels[0], labels[2], labels[4]}) == 3
    assert louvain(*csr_of(5, e2))[0].tolist() == labels.tolist()


def test_empty_and_edgeless_graphs():
    assert oc.louvain(np.zeros(1, np.int64), [], [])[0].tolist() == []
    got, levels = louvain(np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0))
    assert got.tolist() == [] and levels == 0
    got, levels = louvain(np.zeros(4, np.int64), np.zeros(0, np.int32), np.zeros(0))      # 3 nodes, no edge
    assert got.tolist() == [1, 2, 3] and levels == 0
    assert oc.oracle_find_clones(np.zeros((2, 3, 5), np.uint32))[0].tolist() == [0] * 5


def test_oracle_pipeline_finds_planted_clones():
    counts = clone_counts(40, 9, seed=5)
    labels, info = oc.oracle_find_clones(counts, k=10)
    assert (labels > 0).all()
    groups = [set(labels[c * 40:(c + 1) * 40].tolist()) for c in range(3)]
    assert sum(len(g) for g in groups) == len(set.union(*groups))       # no clone mixes planted clones


# ---------------------------------------------------------------------------------------------------------------- library
@pytest.mark.parametrize("seed,n_per,V,k,res", [(1, 30, 6, 10, 1.0), (2, 70, 16, 5, 1.0), (3, 50, 12, 20, 0.5),
                                                (4, 40, 7, 2, 2.0), (5, 100, 30, 10, 1.0)])
def test_louvain_host_equals_oracle(seed, n_per, V, k, res):
    counts = clone_counts(n_per, V, seed, noise=0.1)
    x = oc.allele_frequencies(counts)
    rows = oc.graph_rows(x)
    nbr, _ = oc.knn(np.ascontiguousarray(x[:, rows].T), k)
    w = oc.snn_weights(nbr)
    csr = oc.snn_graph(nbr, w)
    mine = snn_graph(nbr, w)
    for a, b in zip(mine, csr):
        np.testing.assert_array_equal(a, b)
    want, levels = oc.louvain(*csr, res)
    got, got_levels = louvain(*csr, res)
    np.testing.assert_array_equal(got, want)
    assert got_levels == levels


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_louvain_host_random_graphs(seed):
    rng = np.random.default_rng(seed)
    n = 150
    e = {}
    for _ in range(600):
        i, j = sorted(rng.integers(0, n, 2).tolist())
        e[(i, j)] = float(rng.integers(1, 20)) / 7.0
    csr = csr_of(n, e)
    want, levels = oc.louvain(*csr, 1.0)
    got, got_levels = louvain(*csr, 1.0)
    np.testing.assert_array_equal(got, want)
    assert got_levels == levels


def test_louvain_host_rejects_bad_graphs():
    from mgatk2_b200 import _lib
    indptr, indices, weights = csr_of(3, {(0, 1): 1.0})
    with pytest.raises(ValueError):
        louvain(indptr, indices, weights, 0.0)
    with pytest.raises(ValueError):
        louvain(indptr, np.array([0, 5], np.int32), weights)
    with pytest.raises(ValueError):
        louvain(indptr, indices, -weights)
    with pytest.raises(ValueError):
        louvain(np.array([1, 1, 2, 2]), indices, weights)
    assert _lib.load().mgatk_louvain_host(-1, None, None, None, 1.0, None, None) == 1


# ---------------------------------------------------------------------------------------------------------------- files
def test_files_round_trip(tmp_path):
    counts = clone_counts(10, 4, seed=9)
    C = counts.shape[2]
    labels, info = oc.oracle_find_clones(counts, k=5)
    labels[3] = 0
    selected = np.ones(C, bool)
    selected[7] = False
    labels[7] = 0
    res = CloneResult(labels, selected, info["rows"], info["nbr"], info["sim"], *info["csr"], info["levels"],
                      np.arange(4, dtype=np.int32) * 5, ["1A>C", "2C>G", "3G>T", "4T>A"])
    barcodes = [f"BC{i:03d}-1" for i in range(C)]
    write_clones(res, barcodes, tmp_path / "clones.tsv.gz")
    names, back = read_clones(tmp_path / "clones.tsv.gz")
    assert names == [b for b, s in zip(barcodes, selected) if s]
    np.testing.assert_array_equal(back, labels[selected])
    table = clone_variant_table(res, counts)
    assert table.dtype == CLONE_VARIANTS_DTYPE and len(table) == res.n_clones * 4
    assert table["n_cells"][::4].sum() == (labels > 0).sum()
    write_clone_variants(table, tmp_path / "clone_variants.tsv.gz")
    t2 = read_clone_variants(tmp_path / "clone_variants.tsv.gz")
    for f in ("clone", "variant", "n_cells", "n_cells_detected"):
        np.testing.assert_array_equal(t2[f], table[f])
    np.testing.assert_allclose(t2["mean_heteroplasmy"], table["mean_heteroplasmy"], rtol=1e-9)
