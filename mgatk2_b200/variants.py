"""Variant statistics: per-variant heteroplasmy statistics and per-cell allele counts, computed on the GPU from the count
planes of a result (DESIGN §8 "Variant statistics"; the semantics of Signac's `IdentifyVariants`, the successor of mgatk
v1's `call` step).

    sums = variant_sums(result)              # mgatk_variant_stats_device: exact integer sums, dev_sum / dev_sq
    table = finalize(sums, n_cells)          # host floats: mean, variance, vmr, strand correlation, ...
    called = call_variants(table)            # n_conf_detected >= 5, strand_correlation >= 0.65, vmr > 0.01
    counts = variant_cells(result, called)   # mgatk_variant_cells_device: uint32 [variants, 3, cells]

`result` is a host `PileupResult` (planes, overflow list and base totals are uploaded to one GPU) or a
`(DeviceOutputs, params)` pair of the resident and streamed paths (nothing is downloaded but the sums). The cells are
those with a QC row (`PileupResult.alive()`) unless `cells` says otherwise; `n_cells` of `finalize` is their number.
"""
from __future__ import annotations

import ctypes
import gzip
import math
from pathlib import Path

import numpy as np

from ._lib import OutputsC, VariantSumsC
from .engine import CELL_QC_DTYPE, OVERFLOW_DTYPE, STATS_FIELDS, PileupResult
from .exceptions import ProcessingError

BASES = "ACGT"
OVER_THRESHOLDS = (5, 10, 20, 95)          # n_cells_over_<k>: cells with d > 0 and a / d >= k / 100

VARIANT_SUMS_DTYPE = np.dtype([
    ("sum_fwd", "<u8"), ("sum_rev", "<u8"), ("sum_cov", "<u8"), ("sum_ff", "<u8"), ("sum_rr", "<u8"), ("sum_fr", "<u8"),
    ("max_alt", "<u8"), ("max_cov", "<u8"), ("dev_sum", "<f8"), ("dev_sq", "<f8"),
    ("n_covered", "<u4"), ("n_detected", "<u4"), ("n_conf_detected", "<u4"), ("n_strand", "<u4"), ("n_over", "<u4", (4,)),
    ("n_low", "<u4"), ("ref", "<i4"), ("valid", "<i4"), ("reserved", "<i4")])
assert VARIANT_SUMS_DTYPE.itemsize == ctypes.sizeof(VariantSumsC) == 128

VARIANT_TABLE_DTYPE = np.dtype([
    ("variant", "U24"), ("position", "<i8"), ("nucleotide", "U3"), ("ref", "U1"), ("alt", "U1"),
    ("n_cells_conf_detected", "<i8"), ("n_cells_detected", "<i8"), ("n_cells_covered", "<i8"),
    ("n_cells_over_5", "<i8"), ("n_cells_over_10", "<i8"), ("n_cells_over_20", "<i8"), ("n_cells_over_95", "<i8"),
    ("n_cells_low_coverage", "<i8"), ("strand_correlation", "<f8"), ("mean", "<f8"), ("variance", "<f8"), ("vmr", "<f8"),
    ("mean_coverage", "<f8"), ("max_heteroplasmy", "<f8")])
_FLOAT_COLUMNS = ("strand_correlation", "mean", "variance", "vmr", "mean_coverage", "max_heteroplasmy")
SUM_COV_LIMIT = 1 << 32                    # sum_cov below this keeps every u64 sum exact (sum f*f <= sum_cov^2)


# ---------------------------------------------------------------------------------------------------------------- floats
def strand_correlation(n: int, sx: int, sy: int, sxx: int, syy: int, sxy: int) -> float:
    """Pearson's r of (forward, reverse) over the n cells with a > 0, from exact integer sums; NaN when n < 2 or a strand
    is constant over those cells."""
    n, sx, sy, sxx, syy, sxy = (int(v) for v in (n, sx, sy, sxx, syy, sxy))
    if n < 2:
        return math.nan
    dx, dy = n * sxx - sx * sx, n * syy - sy * sy
    if dx == 0 or dy == 0:
        return math.nan
    return (n * sxy - sx * sy) / math.sqrt(float(dx * dy))


def variant_mean(sum_fwd, sum_rev, sum_cov) -> np.ndarray:
    """(sum_fwd + sum_rev) / sum_cov, 0 where sum_cov = 0 (the mean the device centres dev_sum / dev_sq on)."""
    alt = (np.asarray(sum_fwd, np.uint64) + np.asarray(sum_rev, np.uint64)).astype(np.float64)
    cov = np.asarray(sum_cov, np.uint64).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(cov > 0, alt / np.where(cov > 0, cov, 1.0), 0.0)


def finalize(sums: np.ndarray, n_cells: int) -> np.ndarray:
    """The host floats of every valid variant of `sums` (VARIANT_SUMS_DTYPE, [P, 4]), positions ascending, then alt
    A, C, G, T. `n_cells` is N, the number of selected cells.
        mean = (sum_fwd + sum_rev) / sum_cov (0 when sum_cov = 0)
        variance = (dev_sq - dev_sum^2 / N) / (N - 1)            NaN when N < 2
        vmr = variance / (mean + 1e-11)
        strand_correlation: Pearson's r over the n_strand cells   NaN when n_strand < 2 or a strand is constant
        max_heteroplasmy = max_alt / max_cov                      NaN when no cell is covered
        mean_coverage = sum_cov / N                               NaN when N = 0
    Raises ProcessingError when a position's sum_cov reaches 2^32 (the u64 sums could have wrapped)."""
    s = np.asarray(sums, VARIANT_SUMS_DTYPE).reshape(-1, 4)
    if len(s) and int(s["sum_cov"].max()) >= SUM_COV_LIMIT:
        raise ProcessingError("variant statistics: a position's summed coverage reaches 2^32")
    pos, alt = np.nonzero(s["valid"] != 0)
    v = s[pos, alt]
    n = int(n_cells)
    t = np.zeros(len(v), VARIANT_TABLE_DTYPE)
    ref = np.array(list(BASES))[np.clip(v["ref"], 0, 3)]
    alts = np.array(list(BASES))[alt]
    t["position"] = pos + 1
    t["ref"], t["alt"] = ref, alts
    t["nucleotide"] = np.char.add(np.char.add(ref, ">"), alts) if len(v) else t["nucleotide"]
    t["variant"] = np.char.add(t["position"].astype(str), t["nucleotide"]) if len(v) else t["variant"]
    t["n_cells_conf_detected"] = v["n_conf_detected"]
    t["n_cells_detected"] = v["n_detected"]
    t["n_cells_covered"] = v["n_covered"]
    for k, thr in enumerate(OVER_THRESHOLDS):
        t[f"n_cells_over_{thr}"] = v["n_over"][:, k]
    t["n_cells_low_coverage"] = v["n_low"]
    mean = variant_mean(v["sum_fwd"], v["sum_rev"], v["sum_cov"])
    t["mean"] = mean
    with np.errstate(divide="ignore", invalid="ignore"):
        var = (v["dev_sq"] - v["dev_sum"] * v["dev_sum"] / n) / (n - 1) if n >= 2 else np.full(len(v), np.nan)
        t["variance"] = var
        t["vmr"] = var / (mean + 1e-11)
        t["mean_coverage"] = v["sum_cov"].astype(np.float64) / n if n >= 1 else np.nan
        t["max_heteroplasmy"] = np.where(v["max_cov"] > 0, v["max_alt"].astype(np.float64) / np.maximum(v["max_cov"], 1), np.nan)
    t["strand_correlation"] = [strand_correlation(*row) for row in
                               zip(v["n_strand"].tolist(), v["sum_fwd"].tolist(), v["sum_rev"].tolist(),
                                   v["sum_ff"].tolist(), v["sum_rr"].tolist(), v["sum_fr"].tolist())]
    return t


def call_mask(table: np.ndarray, min_conf_detected: int = 5, min_strand_correlation: float = 0.65,
              min_vmr: float = 0.01) -> np.ndarray:
    """Signac's documented filter: n_cells_conf_detected >= 5, strand_correlation >= 0.65, vmr > 0.01 (NaN fails)."""
    with np.errstate(invalid="ignore"):
        return ((table["n_cells_conf_detected"] >= min_conf_detected) & (table["strand_correlation"] >= min_strand_correlation)
                & (table["vmr"] > min_vmr))


def call_variants(table: np.ndarray, min_conf_detected: int = 5, min_strand_correlation: float = 0.65,
                  min_vmr: float = 0.01) -> np.ndarray:
    """The rows of `table` that pass `call_mask`."""
    return table[call_mask(table, min_conf_detected, min_strand_correlation, min_vmr)]


# ---------------------------------------------------------------------------------------------------------------- device
class _Source:
    """A result on one GPU: the C-ABI view (params, outputs), its row count and its QC rows on the host."""

    def __init__(self, source, engine):
        import torch
        from .pileup import get_engine
        if isinstance(source, PileupResult):
            self.engine = engine or get_engine(0)
            dev = torch.device("cuda", self.engine.device)
            res = source
            C, P = len(res.planes), int(res.mito_length)
            stats = np.zeros(len(STATS_FIELDS), np.uint64)
            stats[STATS_FIELDS.index("n_overflow")] = len(res.overflow)
            ovf = np.ascontiguousarray(res.overflow, OVERFLOW_DTYPE)
            self._keep = [torch.from_numpy(np.ascontiguousarray(res.planes)).to(dev),
                          torch.from_numpy(stats.view(np.int64)).to(dev),
                          torch.from_numpy(np.ascontiguousarray(res.base_totals, np.int64)).to(dev),
                          torch.from_numpy(ovf.view(np.uint8).reshape(-1) if len(ovf) else np.zeros(1, np.uint8)).to(dev)]
            planes, st, bt, ov = self._keep
            self.outputs = OutputsC(planes.data_ptr(), None, st.data_ptr(), bt.data_ptr(),
                                    ov.data_ptr() if len(ovf) else None, len(ovf))
            self.params = _params(C, P)
            self.qc, self.min_reads = res.cell_qc, res.min_reads_per_cell
            self.columns = None if res.columns is None else np.asarray(res.columns)
        else:
            dout, params = source
            self.engine = engine or get_engine(dout.planes.device.index)
            torch.cuda.synchronize(self.engine.device)
            stats_np = dout.stats.cpu().numpy().view(np.uint64)
            rc = self.engine.lib.mgatk_check_stats(stats_np.ctypes.data)
            if rc:
                self.engine._raise(rc)
            if int(stats_np[STATS_FIELDS.index("n_overflow")]) > dout.overflow_capacity:
                raise ProcessingError("variant statistics: the result's overflow list is incomplete")
            C, P = int(dout.n_cells), int(params.mito_length)
            self.outputs = self.engine._outputs_c(dout)
            self.params = _params(C, P)
            self.qc = dout.cell_qc.cpu().numpy().view(CELL_QC_DTYPE)[:C]
            self.min_reads = int(params.min_reads_per_cell)
            self.columns = None
        self.n_cells, self.mito_length = C, P

    def alive(self) -> np.ndarray:
        n = self.qc["n_reads"].astype(np.int64)
        return (n >= max(1, self.min_reads)) & (self.qc["sum_depth"] > 0)

    def barcodes(self, barcode_list) -> list:
        """The name of every row: barcode_list[columns[k]] (row k is whitelist entry k without columns)."""
        rows = range(self.n_cells) if self.columns is None else self.columns.tolist()
        return [barcode_list[int(c)] for c in rows]

    def stream(self):
        import torch
        return ctypes.c_void_p(torch.cuda.current_stream(self.engine.device).cuda_stream)


def _params(n_cells: int, mito_length: int):
    from ._lib import ParamsC
    p = ParamsC()
    p.n_cells, p.mito_length = int(n_cells), int(mito_length)
    return p


def cell_mask(n_cells: int, cells) -> np.ndarray:
    """bool [n_cells] from a bool mask or a list of row indices."""
    c = np.asarray(cells)
    if c.dtype == bool:
        if c.shape != (n_cells,):
            raise ValueError(f"cell mask of shape {c.shape}, expected ({n_cells},)")
        return c.copy()
    m = np.zeros(n_cells, bool)
    if len(c):
        if c.min() < 0 or c.max() >= n_cells:
            raise ValueError("cell index out of range")
        m[c.astype(np.int64)] = True
    return m


def selected_cells(source, cells=None, engine=None) -> np.ndarray:
    """The bool row mask variant_sums uses for `cells` (default: the cells with a QC row)."""
    src = source if isinstance(source, _Source) else _Source(source, engine)
    return src.alive() if cells is None else cell_mask(src.n_cells, cells)


def variant_sums(source, engine=None, cells=None, low_coverage_threshold: int = 10) -> np.ndarray:
    """VARIANT_SUMS_DTYPE [P, 4] of `source` over the selected cells (mgatk_variant_stats_device)."""
    import torch
    src = source if isinstance(source, _Source) else _Source(source, engine)
    mask = selected_cells(src, cells)
    dev = torch.device("cuda", src.engine.device)
    mask_t = torch.from_numpy(mask.astype(np.uint8)).to(dev) if src.n_cells else None
    out = torch.empty(max(src.mito_length, 1) * 4 * VARIANT_SUMS_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    rc = src.engine.lib.mgatk_variant_stats_device(src.engine.handle, ctypes.byref(src.params), ctypes.byref(src.outputs),
                                                   mask_t.data_ptr() if mask_t is not None else None,
                                                   int(low_coverage_threshold), out.data_ptr(), src.stream())
    if rc:
        src.engine._raise(rc)
    sums = out.cpu().numpy().view(VARIANT_SUMS_DTYPE)[: src.mito_length * 4].reshape(src.mito_length, 4).copy()
    if len(sums) and int(sums["sum_cov"].max()) >= SUM_COV_LIMIT:
        raise ProcessingError("variant statistics: a position's summed coverage reaches 2^32")
    return sums


def variant_ids(variants) -> np.ndarray:
    """int32 ids pos * 4 + alt (0-based pos) from an id array or a table of finalize (1-based `position`, `alt`)."""
    v = np.asarray(variants)
    if v.dtype.names:
        return ((v["position"].astype(np.int64) - 1) * 4 + np.array([BASES.index(a) for a in v["alt"].tolist()], np.int64)
                ).astype(np.int32)
    return v.astype(np.int32).reshape(-1)


def variant_cells_device(source, variants, engine=None):
    """The counts of variant_cells left on the GPU: a torch int32 tensor [n_variants, 3, n_cells] holding the uint32
    values (enqueued on the current stream)."""
    import torch
    src = source if isinstance(source, _Source) else _Source(source, engine)
    ids = variant_ids(variants)
    if len(ids) and (ids.min() < 0 or ids.max() >= 4 * src.mito_length):
        raise ValueError("variant id outside [0, 4 * mito_length)")
    dev = torch.device("cuda", src.engine.device)
    n = len(ids)
    ids_t = torch.from_numpy(ids.copy() if n else np.zeros(1, np.int32)).to(dev)
    out = torch.empty(max(n * 3 * src.n_cells, 1), dtype=torch.int32, device=dev)
    rc = src.engine.lib.mgatk_variant_cells_device(src.engine.handle, ctypes.byref(src.params), ctypes.byref(src.outputs),
                                                   ids_t.data_ptr(), n, out.data_ptr(), src.stream())
    if rc:
        src.engine._raise(rc)
    return out[: n * 3 * src.n_cells].view(n, 3, src.n_cells)


def variant_cells(source, variants, engine=None) -> np.ndarray:
    """uint32 [n_variants, 3, n_cells]: exact alt forward, alt reverse and coverage of every row of `source` for every
    variant (mgatk_variant_cells_device). `variants` is a table of finalize or int ids pos * 4 + alt."""
    out = variant_cells_device(source, variants, engine)
    return out.cpu().numpy().view(np.uint32).copy()


# ---------------------------------------------------------------------------------------------------------------- files
def _fmt(x) -> str:
    return "NA" if isinstance(x, float) and math.isnan(x) else format(x, ".10g") if isinstance(x, float) else str(x)


def _gzip_text(path: Path, lines):
    with open(path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
        for line in lines:
            f.write(line.encode())


def write_variant_stats(table: np.ndarray, path) -> None:
    """`variant_stats.tsv.gz`: a header line, one row per variant of `table`, floats '.10g', NaN as NA."""
    names = table.dtype.names
    rows = ("\t".join(_fmt(x) for x in row) + "\n" for row in table.tolist())
    _gzip_text(Path(path), ["\t".join(names) + "\n", *rows])


def write_variant_cells(called: np.ndarray, counts: np.ndarray, barcodes, mask: np.ndarray, path) -> None:
    """`variant_cells.tsv.gz`: variant, barcode, alt_fwd, alt_rev, coverage for every called variant and every selected
    row with coverage > 0; `barcodes[k]` names row k, `counts` is variant_cells of `called`."""
    def rows():
        yield "variant\tbarcode\talt_fwd\talt_rev\tcoverage\n"
        for i, name in enumerate(called["variant"].tolist()):
            f, r, d = counts[i]
            for k in np.nonzero(mask & (d > 0))[0].tolist():
                yield f"{name}\t{barcodes[k]}\t{f[k]}\t{r[k]}\t{d[k]}\n"
    _gzip_text(Path(path), rows())


def read_variant_stats(path) -> np.ndarray:
    """A `variant_stats.tsv.gz` back as a table of finalize (NA -> NaN)."""
    with gzip.open(path, "rt") as f:
        header = f.readline().rstrip("\n").split("\t")
        body = [line.rstrip("\n").split("\t") for line in f]
    t = np.zeros(len(body), VARIANT_TABLE_DTYPE)
    for j, name in enumerate(header):
        col = [r[j] for r in body]
        t[name] = [math.nan if x == "NA" else float(x) for x in col] if name in _FLOAT_COLUMNS else col
    return t


def write_variant_files(result, barcode_list, output_dir, engine=None, low_coverage_threshold: int = 10, **call_kwargs):
    """`output_dir/variant_stats.tsv.gz` and `output_dir/variant_cells.tsv.gz` for the cells with a QC row of a host
    result (or a `_Source` of one, so later steps reuse its upload); barcodes are `barcode_list[columns[k]]` for row k.
    Returns the called variants and their counts (variant_cells)."""
    src = result if isinstance(result, _Source) else _Source(result, engine)     # planes uploaded once for both calls
    mask = src.alive()
    sums = variant_sums(src, cells=mask, low_coverage_threshold=low_coverage_threshold)
    table = finalize(sums, int(mask.sum()))
    called = call_variants(table, **call_kwargs)
    counts = variant_cells(src, called)
    out = Path(output_dir)
    write_variant_stats(table, out / "variant_stats.tsv.gz")
    write_variant_cells(called, counts, src.barcodes(barcode_list), mask, out / "variant_cells.tsv.gz")
    return called, counts
