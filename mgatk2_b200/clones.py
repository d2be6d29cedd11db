"""Clones: cells grouped by the heteroplasmy of called mtDNA variants (DESIGN §8 "Clones"; Signac's `AlleleFreq` followed
by `FindClonotypes`, with an exact kNN search where Signac uses Annoy's approximate one, and plain deterministic Louvain
where Seurat's default is SLM with random starts: labels are comparable in kind, not identical to Seurat's).

    clones = find_clones(result)              # variants: call_variants(finalize(variant_sums(result))) by default
    clones.labels                             # int32 [n_cells]: 0 = NA (no called variant detected) or not selected
    table = clone_variants(result, clones)    # per clone x variant: cells, cells detected, mean heteroplasmy

`result` is a host `PileupResult` or a `(DeviceOutputs, params)` pair, as in `variants.py`. The allele counts, the
heteroplasmy matrix and the all-pairs search stay on the GPU (mgatk_clone_knn_device, mgatk_clone_snn_device); the kNN
lists come back to build the SNN graph, and Louvain runs on the host (mgatk_louvain_host).
"""
from __future__ import annotations

import ctypes
import gzip
from dataclasses import dataclass
from pathlib import Path

import numpy as np

from .variants import (BASES, _fmt, _gzip_text, _Source, call_variants, finalize, selected_cells, variant_cells,
                       variant_cells_device, variant_ids, variant_sums)

K_MAX = 64                                  # MGATK_CLONE_K_MAX
CLONE_VARIANTS_DTYPE = np.dtype([("clone", "<i4"), ("variant", "U24"), ("n_cells", "<i8"), ("n_cells_detected", "<i8"),
                                 ("mean_heteroplasmy", "<f8")])


@dataclass
class CloneResult:
    labels: np.ndarray          # int32 [n_cells]: clone number 1..K, 0 = NA or not selected
    selected: np.ndarray        # bool [n_cells]: the selected cells
    rows: np.ndarray            # int32 [n]: the graph rows (cell indices), ascending
    neighbors: np.ndarray       # int32 [n, k_eff]: N(i) as row indices, i first
    similarity: np.ndarray      # fp64 [n, k_eff]: cos(i, j), 1.0 for i itself
    indptr: np.ndarray          # SNN graph, symmetric CSR over the rows: int64 [n + 1]
    indices: np.ndarray         # int32
    weights: np.ndarray         # fp64
    n_levels: int               # Louvain levels whose first phase moved a node
    variants: np.ndarray        # int32 ids pos * 4 + alt of the variants used
    variant_names: list         # their names (`302A>G`; `302>G` when given as ids)

    @property
    def n_clones(self) -> int:
        return int(self.labels.max()) if len(self.labels) else 0


def _names(variants, ids: np.ndarray) -> list:
    v = np.asarray(variants)
    if v.dtype.names:
        return [str(s) for s in v["variant"].tolist()]
    return [f"{int(i) // 4 + 1}>{BASES[int(i) % 4]}" for i in ids.tolist()]


def allele_frequencies(source, variants, engine=None, cells=None) -> np.ndarray:
    """fp64 [n_variants, n_cells]: x = (f + r) / d of every variant and cell (0 where d = 0 and for cells not selected;
    Signac's AlleleFreq) from the exact counts of variant_cells."""
    src = source if isinstance(source, _Source) else _Source(source, engine)
    mask = selected_cells(src, cells)
    x = _heteroplasmy(variant_cells(src, variants))[1]
    x[:, ~mask] = 0.0
    return x


def _heteroplasmy(counts: np.ndarray):
    """(a = f + r as uint64, x = a / d in fp64, 0 where d = 0) of uint32 counts [V, 3, C]."""
    c = np.asarray(counts, np.uint64)
    a, d = c[:, 0] + c[:, 1], c[:, 2].astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return a, np.where(d > 0, a.astype(np.float64) / np.where(d > 0, d, 1.0), 0.0)


def snn_graph(nbr: np.ndarray, w: np.ndarray, prune: float = 1.0 / 15):
    """Symmetric CSR (indptr int64, indices int32 ascending, weights fp64) of the pairs (i, j) with j in N(i) or i in
    N(j), diagonal included, weight w = s / (2 k_eff - s) of the directed kNN edges (the same from either end), pairs with
    w < prune dropped."""
    n, k = nbr.shape
    src = np.repeat(np.arange(n, dtype=np.int64), k)
    dst = nbr.astype(np.int64).reshape(-1)
    ww = w.reshape(-1)
    key = np.concatenate([src * n + dst, dst * n + src])
    wt = np.concatenate([ww, ww])
    key, first = np.unique(key, return_index=True)
    wt = wt[first]
    keep = ~(wt < prune)
    key, wt = key[keep], wt[keep]
    i, j = key // max(n, 1), key % max(n, 1)
    indptr = np.zeros(n + 1, np.int64)
    np.add.at(indptr, i + 1, 1)
    return np.cumsum(indptr).astype(np.int64), j.astype(np.int32), wt.astype(np.float64)


def louvain(indptr, indices, weights, resolution: float = 1.0):
    """(labels int32 [n] in 1..K, levels) of mgatk_louvain_host; needs the library, not a GPU."""
    from . import _lib
    lib = _lib.load()
    indptr = np.ascontiguousarray(indptr, np.int64)
    indices = np.ascontiguousarray(indices, np.int32)
    weights = np.ascontiguousarray(weights, np.float64)
    n = len(indptr) - 1
    labels = np.zeros(max(n, 1), np.int32)
    levels = ctypes.c_int32(0)
    rc = lib.mgatk_louvain_host(n, indptr.ctypes.data, indices.ctypes.data if len(indices) else None,
                                weights.ctypes.data if len(weights) else None, float(resolution), labels.ctypes.data,
                                ctypes.byref(levels))
    if rc:
        raise ValueError(f"mgatk_louvain_host: {lib.mgatk_status_string(rc).decode()}")
    return labels[:n], int(levels.value)


def find_clones(source, variants=None, engine=None, cells=None, k: int = 10, resolution: float = 1.0,
                prune: float = 1.0 / 15) -> CloneResult:
    """Clone labels of the selected cells (default: the cells with a QC row) from the heteroplasmy of `variants` (a
    table of finalize or int ids pos * 4 + alt; default: the variants call_variants keeps over the selected cells).
    Cells without a detected variant get 0 (NA). k in [2, 64]; prune is Seurat's prune.SNN."""
    import torch
    if not 2 <= int(k) <= K_MAX:
        raise ValueError(f"k must be in [2, {K_MAX}]")
    if not resolution > 0:
        raise ValueError("resolution must be positive")
    src = source if isinstance(source, _Source) else _Source(source, engine)
    mask = selected_cells(src, cells)
    if variants is None:
        variants = call_variants(finalize(variant_sums(src, cells=mask), int(mask.sum())))
    ids = variant_ids(variants)
    names = _names(variants, ids)
    C, V = src.n_cells, len(ids)
    dev = torch.device("cuda", src.engine.device)
    rows = np.zeros(0, np.int32)
    if V and C:
        counts = variant_cells_device(src, ids)                           # int32 view of uint32 [V, 3, C], on the GPU
        hit = (((counts[:, 0] != 0) | (counts[:, 1] != 0)) & (counts[:, 2] != 0)).any(dim=0)
        hit &= torch.from_numpy(mask).to(dev)
        rows_t = torch.nonzero(hit).flatten().to(torch.int32)
        rows = rows_t.cpu().numpy()
    n = len(rows)
    k_eff = min(int(k), n)
    if n == 0:
        return CloneResult(np.zeros(C, np.int32), mask, rows, np.zeros((0, 0), np.int32), np.zeros((0, 0)),
                           np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0), 0, ids, names)
    lib, h, stream = src.engine.lib, src.engine.handle, src.stream()
    nbr = torch.empty((n, k_eff), dtype=torch.int32, device=dev)
    sim = torch.empty((n, k_eff), dtype=torch.float64, device=dev)
    w = torch.empty((n, k_eff), dtype=torch.float64, device=dev)
    rc = lib.mgatk_clone_knn_device(h, counts.data_ptr(), rows_t.data_ptr(), n, C, V, int(k), nbr.data_ptr(),
                                    sim.data_ptr(), stream)
    if rc:
        src.engine._raise(rc)
    rc = lib.mgatk_clone_snn_device(h, nbr.data_ptr(), n, k_eff, w.data_ptr(), stream)
    if rc:
        src.engine._raise(rc)
    nbr_h, sim_h, w_h = nbr.cpu().numpy(), sim.cpu().numpy(), w.cpu().numpy()
    indptr, indices, weights = snn_graph(nbr_h, w_h, prune)
    lab, levels = louvain(indptr, indices, weights, resolution)
    labels = np.zeros(C, np.int32)
    labels[rows] = lab
    return CloneResult(labels, mask, rows, nbr_h, sim_h, indptr, indices, weights, levels, ids, names)


def clone_variant_table(clones: CloneResult, counts: np.ndarray) -> np.ndarray:
    """CLONE_VARIANTS_DTYPE, clones ascending then variants in order: the clone's cells, those with a > 0 and the mean of
    x = (f + r) / d over the clone's cells; `counts` is variant_cells of clones.variants."""
    a, x = _heteroplasmy(counts)
    K, V = clones.n_clones, len(clones.variants)
    t = np.zeros(K * V, CLONE_VARIANTS_DTYPE)
    for q in range(1, K + 1):
        members = clones.labels == q
        s = slice((q - 1) * V, q * V)
        t["clone"][s] = q
        t["variant"][s] = clones.variant_names
        t["n_cells"][s] = int(members.sum())
        t["n_cells_detected"][s] = (a[:, members] > 0).sum(axis=1)
        t["mean_heteroplasmy"][s] = x[:, members].mean(axis=1)
    return t


def clone_variants(source, clones: CloneResult, engine=None) -> np.ndarray:
    """Per clone x variant of `clones`: n_cells, n_cells_detected (a > 0) and mean_heteroplasmy."""
    return clone_variant_table(clones, variant_cells(source, clones.variants, engine))


# ---------------------------------------------------------------------------------------------------------------- files
def write_clones(clones: CloneResult, barcodes, path) -> None:
    """`clones.tsv.gz`: barcode, clone for every selected row (NA for a row without a clone); `barcodes[k]` names row k."""
    rows = np.nonzero(clones.selected)[0].tolist()
    lab = clones.labels
    _gzip_text(Path(path), ["barcode\tclone\n", *(f"{barcodes[k]}\t{lab[k] if lab[k] else 'NA'}\n" for k in rows)])


def read_clones(path):
    """A `clones.tsv.gz` back: (barcodes, int32 clone numbers with 0 for NA)."""
    with gzip.open(path, "rt") as f:
        f.readline()
        body = [line.rstrip("\n").split("\t") for line in f]
    return [b for b, _ in body], np.array([0 if c == "NA" else int(c) for _, c in body], np.int32)


def write_clone_variants(table: np.ndarray, path) -> None:
    """`clone_variants.tsv.gz`: a header line, one row per clone x variant, floats '.10g'."""
    rows = ("\t".join(_fmt(x) for x in row) + "\n" for row in table.tolist())
    _gzip_text(Path(path), ["\t".join(table.dtype.names) + "\n", *rows])


def read_clone_variants(path) -> np.ndarray:
    with gzip.open(path, "rt") as f:
        header = f.readline().rstrip("\n").split("\t")
        body = [line.rstrip("\n").split("\t") for line in f]
    t = np.zeros(len(body), CLONE_VARIANTS_DTYPE)
    for j, name in enumerate(header):
        t[name] = [r[j] for r in body]
    return t


def write_clone_files(source, barcode_list, output_dir, called, counts, **find_kwargs) -> CloneResult:
    """`output_dir/clones.tsv.gz` and `output_dir/clone_variants.tsv.gz` for the cells with a QC row of `source` (the
    `_Source` write_variant_files used), from the variants `called` and their host counts; barcodes are
    `barcode_list[columns[k]]` for row k."""
    clones = find_clones(source, called, **find_kwargs)
    out = Path(output_dir)
    write_clones(clones, source.barcodes(barcode_list), out / "clones.tsv.gz")
    write_clone_variants(clone_variant_table(clones, counts), out / "clone_variants.tsv.gz")
    return clones
