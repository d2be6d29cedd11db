"""Clone markers: the variants that distinguish each group of cells from the rest (DESIGN §8 "Clone markers"; Seurat's
`FindAllMarkers` with its default two-sided Wilcoxon rank-sum test on the allele-frequency assay, one group against the
other cells).

    clones = find_clones(result)
    table = clone_markers(result, clones)               # per clone x variant: auc, U, p, Bonferroni p, ...
    table = find_markers(result, labels, variants)      # any labelling: 1..G a group, anything else left out

`result` is a host `PileupResult` or a `(DeviceOutputs, params)` pair, as in `variants.py`. The counts stay on the GPU,
where mgatk_marker_ranks_device ranks x = (f + r) / d per variant and returns exact integer rank sums and tie terms;
the host forms the test statistics from them (`wilcoxon`).
"""
from __future__ import annotations

import gzip
import math
from pathlib import Path

import numpy as np

from .clones import _heteroplasmy, _names
from .exceptions import ProcessingError
from .variants import _fmt, _gzip_text, _Source, variant_cells_device, variant_ids

MAX_CELLS = 1 << 21                         # MGATK_MARKER_MAX_CELLS: the population N, so that N^3 stays below 2^63
_FIELDS = [("variant", "U24"), ("n_cells", "<i8"), ("n_cells_rest", "<i8"), ("n_cells_detected", "<i8"),
           ("n_cells_detected_rest", "<i8"), ("mean_heteroplasmy", "<f8"), ("mean_heteroplasmy_rest", "<f8"),
           ("auc", "<f8"), ("statistic", "<f8"), ("p_value", "<f8"), ("p_value_adj", "<f8")]
MARKERS_DTYPE = np.dtype([("group", "<i4"), *_FIELDS])
CLONE_MARKERS_DTYPE = np.dtype([("clone", "<i4"), *_FIELDS])


def wilcoxon(rank2: int, ties: int, n1: int, N: int):
    """(U, auc, z, p) of one group of n1 cells in a population of N from the exact integers of the device: rank2 = the
    sum of 2 * mid-rank over the group, ties = the sum of t^3 - t over runs of equal values. R's
    `wilcox.test(exact = FALSE, correct = TRUE)`:
        U = rank2 / 2 - n1 (n1 + 1) / 2,  auc = U / (n1 n2),  mu = n1 n2 / 2
        sigma^2 = n1 n2 / 12 ((N + 1) - ties / (N (N - 1))),  z = (U - mu - sign(U - mu) / 2) / sigma
        p = erfc(|z| / sqrt(2)), at most 1
    auc, z and p are NaN when n1 = 0, n2 = 0 or sigma = 0 (every value tied)."""
    rank2, ties, n1, N = int(rank2), int(ties), int(n1), int(N)
    n2 = N - n1
    twice_u = rank2 - n1 * (n1 + 1)                         # 2 U, exact
    U = twice_u / 2
    if n1 <= 0 or n2 <= 0:
        return U, math.nan, math.nan, math.nan
    prod = n1 * n2
    var = prod / 12 * ((N + 1) - ties / (N * (N - 1)))
    if not var > 0:
        return U, math.nan, math.nan, math.nan
    d2 = twice_u - prod                                     # 2 (U - mu), exact
    num = (d2 - (d2 > 0) + (d2 < 0)) / 2                    # U - mu - sign(U - mu) / 2
    z = num / math.sqrt(var)
    return U, U / prod, z, min(1.0, math.erfc(abs(z) / math.sqrt(2.0)))


def bonferroni(p, n_tests: int) -> np.ndarray:
    """Seurat's adjustment over the features tested: min(1, p * n_tests); NaN stays NaN."""
    return np.minimum(1.0, np.asarray(p, np.float64) * n_tests)


def device_ranks(src: _Source, counts_dev, labels: np.ndarray, n_groups: int):
    """(rank2 uint64 [V, G], ties uint64 [V]) of mgatk_marker_ranks_device for the int32 labels of the source's rows."""
    import torch
    V, C = int(counts_dev.shape[0]), src.n_cells
    dev = torch.device("cuda", src.engine.device)
    lab_t = torch.from_numpy(np.ascontiguousarray(labels, np.int32) if C else np.zeros(1, np.int32)).to(dev)
    rank2 = torch.empty(max(V * n_groups, 1), dtype=torch.int64, device=dev)
    ties = torch.empty(max(V, 1), dtype=torch.int64, device=dev)
    rc = src.engine.lib.mgatk_marker_ranks_device(src.engine.handle, counts_dev.data_ptr() if V and C else None,
                                                  lab_t.data_ptr(), C, V, int(n_groups), rank2.data_ptr(),
                                                  ties.data_ptr(), src.stream())
    if rc:
        src.engine._raise(rc)
    return (rank2.cpu().numpy().view(np.uint64)[: V * n_groups].reshape(V, n_groups),
            ties.cpu().numpy().view(np.uint64)[:V].copy())


def _table(src: _Source, labels, ids: np.ndarray, names: list, counts, dtype) -> np.ndarray:
    lab = np.asarray(labels)
    if lab.shape != (src.n_cells,):
        raise ValueError(f"labels of shape {lab.shape}, expected ({src.n_cells},)")
    lab = lab.astype(np.int64)
    G = int(lab.max()) if lab.size else 0
    if G > src.n_cells:
        raise ValueError("group numbers run from 1 to at most the number of cells")
    V = len(ids)
    if G < 1:
        return np.zeros(0, dtype)
    inside = lab >= 1
    N = int(inside.sum())
    if N > MAX_CELLS:
        raise ProcessingError(f"clone markers: {N} cells in the test, at most 2^21")
    lab32 = np.where(inside, lab, 0).astype(np.int32)
    counts_dev = variant_cells_device(src, ids)
    rank2, ties = device_ranks(src, counts_dev, lab32, G)
    if counts is None:
        counts = counts_dev.cpu().numpy().view(np.uint32)
    a, x = _heteroplasmy(counts)
    t = np.zeros(G * V, dtype)
    key = dtype.names[0]
    for g in range(1, G + 1):
        members = lab == g
        rest = inside & ~members
        n1 = int(members.sum())
        s = slice((g - 1) * V, g * V)
        t[key][s] = g
        t["variant"][s] = names
        t["n_cells"][s] = n1
        t["n_cells_rest"][s] = N - n1
        t["n_cells_detected"][s] = (a[:, members] > 0).sum(axis=1)
        t["n_cells_detected_rest"][s] = (a[:, rest] > 0).sum(axis=1)
        t["mean_heteroplasmy"][s] = x[:, members].mean(axis=1) if n1 else math.nan
        t["mean_heteroplasmy_rest"][s] = x[:, rest].mean(axis=1) if N - n1 else math.nan
        stats = [wilcoxon(rank2[v, g - 1], ties[v], n1, N) for v in range(V)]
        t["statistic"][s] = [u for u, _, _, _ in stats]
        t["auc"][s] = [auc for _, auc, _, _ in stats]
        t["p_value"][s] = [p for _, _, _, p in stats]
    t["p_value_adj"] = bonferroni(t["p_value"], V)
    return t


def find_markers(source, labels, variants, engine=None, counts=None) -> np.ndarray:
    """MARKERS_DTYPE, groups ascending then `variants` in order: each group g in 1..G (G = the largest label) against the
    other cells with a label in [1, G]; a cell labelled 0 or below is not in the test. `variants` is a table of finalize
    or int ids pos * 4 + alt; `counts`, when given, are their host counts (variant_cells), used for the descriptive
    columns instead of downloading them. Every variant is tested: there are no prefilters."""
    src = source if isinstance(source, _Source) else _Source(source, engine)
    ids = variant_ids(variants)
    return _table(src, labels, ids, _names(variants, ids), counts, MARKERS_DTYPE)


def clone_markers(source, clones, engine=None, counts=None) -> np.ndarray:
    """CLONE_MARKERS_DTYPE: find_markers of every clone of `clones` (a CloneResult) against the other graph cells on
    the clones' variants; NA cells (label 0) are not in the test."""
    src = source if isinstance(source, _Source) else _Source(source, engine)
    return _table(src, clones.labels, np.asarray(clones.variants, np.int32), list(clones.variant_names), counts,
                  CLONE_MARKERS_DTYPE)


# ---------------------------------------------------------------------------------------------------------------- files
def _fmt_u(u: float) -> str:
    """U exactly: an integer or an integer plus one half."""
    return str(int(u)) if u == int(u) else format(u, ".1f")


def write_clone_markers(table: np.ndarray, path) -> None:
    """`clone_markers.tsv.gz`: a header line, one row per clone x variant, floats '.10g', NaN as NA, U exact."""
    names = table.dtype.names
    k = names.index("statistic")
    rows = ("\t".join(_fmt_u(x) if j == k else _fmt(x) for j, x in enumerate(row)) + "\n" for row in table.tolist())
    _gzip_text(Path(path), ["\t".join(names) + "\n", *rows])


def read_clone_markers(path) -> np.ndarray:
    """A `clone_markers.tsv.gz` back as CLONE_MARKERS_DTYPE (NA -> NaN)."""
    with gzip.open(path, "rt") as f:
        header = f.readline().rstrip("\n").split("\t")
        body = [line.rstrip("\n").split("\t") for line in f]
    t = np.zeros(len(body), CLONE_MARKERS_DTYPE)
    for j, name in enumerate(header):
        col = [r[j] for r in body]
        t[name] = [math.nan if x == "NA" else float(x) for x in col] if t.dtype[name].kind == "f" else col
    return t

