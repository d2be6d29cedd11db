"""Large mtDNA deletions on the GPU (DESIGN §8 "Deletions"): the breakpoints mgatk-del-find finds from soft-clipped
reads, and per cell the junction reads against the reads that span a breakpoint, as mgatk-del counts them.

    scan = scan_deletions(parts, config, n_cells, deletions=[(8470, 13446)], find=True)   # one pass over the reads
    cands = find_deletions(scan, result.reference_alleles())                               # breakpoint pairs
    table = deletion_heteroplasmy(scan, cells=result.alive())                              # per cell and deletion

Deletions are given as HGVS-style 1-based ranges of the deleted positions, (first, last) = m.{first}_{last}del; inside,
a deletion is (l, r) = (first - 2, last): the last kept position before and the first kept position after the deleted
segment, 0-based. The reads are those the pileup counts (stage 1, dedup, mapq); the device returns exact integers
(`mgatk_deletion_scan_device`) and heteroplasmy = del / (del + wt) is formed here, NaN when del + wt = 0."""
from __future__ import annotations

import ctypes
import gzip
import math
from dataclasses import dataclass
from pathlib import Path

import numpy as np

from .batch import ReadBatch
from .exceptions import PileupKernelError
from .variants import _fmt, _gzip_text

DEL_KMER = 16                      # MGATK_DEL_KMER: clipped bases per breakpoint in the consensus histograms
DEL_MAX = 1024                     # MGATK_DEL_MAX: deletions per scan
CLASSES = ("clip_left", "clip_right", "gap", "wt")

CANDIDATES_DTYPE = np.dtype([("l", "<i4"), ("r", "<i4"), ("deletion", "U32"), ("first", "<i4"), ("last", "<i4"),
                             ("length", "<i4"), ("support", "U5"), ("reads_left", "<u8"), ("reads_right", "<u8"),
                             ("consensus_left", f"U{DEL_KMER}"), ("consensus_right", f"U{DEL_KMER}")])
HETEROPLASMY_DTYPE = np.dtype([("cell", "<i4"), ("deletion", "U32"), ("index", "<i4"), ("clip_left", "<u4"),
                               ("clip_right", "<u4"), ("gap", "<u4"), ("wt", "<u4"), ("heteroplasmy", "<f8")])


def hgvs_to_breakpoints(first: int, last: int) -> tuple[int, int]:
    """1-based deleted range (first, last) -> (l, r), 0-based kept positions around it."""
    return int(first) - 2, int(last)


def breakpoints_to_hgvs(l: int, r: int) -> tuple[int, int]:
    return int(l) + 2, int(r)


def deletion_name(l: int, r: int) -> str:
    first, last = breakpoints_to_hgvs(l, r)
    return f"m.{first}_{last}del"


def breakpoints(deletions) -> np.ndarray:
    """int32 [D, 2] (l, r) of 1-based (first, last) ranges, or of a table with fields `l` and `r` (find_deletions)."""
    if deletions is None:
        return np.zeros((0, 2), np.int32)
    if isinstance(deletions, np.ndarray) and deletions.dtype.names and "l" in deletions.dtype.names:
        return np.stack([deletions["l"], deletions["r"]], axis=1).astype(np.int32).reshape(-1, 2)
    return np.array([hgvs_to_breakpoints(f, t) for f, t in deletions], np.int32).reshape(-1, 2)


@dataclass
class DeletionScan:
    """Exact integers of one scan. `counts[d, k, c]`: reads of cell c in class CLASSES[k] for deletion d = (l, r) =
    deletions[d]. The histograms (None without discovery): end_clip[p] / start_clip[p] reads with a trailing / leading
    clip of at least min_clip ending / starting at p, end_seq / start_seq [P, DEL_KMER, 4] their clipped bases (A, C, G, T)
    by distance from the junction."""
    deletions: np.ndarray
    counts: np.ndarray
    end_clip: np.ndarray | None
    start_clip: np.ndarray | None
    end_seq: np.ndarray | None
    start_seq: np.ndarray | None
    mito_length: int
    min_clip: int


def scan_deletions(batches, config, n_cells: int, deletions=None, find: bool = False, device: int = 0,
                   min_clip: int = 5) -> DeletionScan:
    """One pass over `batches` (a ReadBatch or an iterable of parts cut on reference_start borders, in file order; their
    bc_idx are columns 0..n_cells-1) on GPU `device`: the class counts of `deletions` (1-based ranges or a
    find_deletions table) and, with `find`, the discovery histograms. `config` (PipelineConfig) gives dedup, min_mapq
    and mito_length. Raises PileupKernelError as the pileup does (unsorted records, a read beyond its extent)."""
    return _scan(batches, config, n_cells, breakpoints(deletions), find, device, min_clip)


def _scan(batches, config, n_cells: int, lr: np.ndarray, find: bool, device: int, min_clip: int = 5) -> DeletionScan:
    import torch

    from .pileup import get_engine
    D, P, K = len(lr), int(config.mito_length), DEL_KMER
    if D > DEL_MAX:
        raise ValueError(f"at most {DEL_MAX} deletions per scan, got {D}")
    bad = ~((lr[:, 0] >= 0) & (lr[:, 0] + 1 < lr[:, 1]) & (lr[:, 1] < P)) if D else np.zeros(0, bool)
    if bad.any():
        raise ValueError(f"deletion outside the contig: {deletion_name(*lr[np.argmax(bad)])}")
    eng = get_engine(device)
    lib = eng.lib
    dev = torch.device("cuda", eng.device)
    if isinstance(batches, ReadBatch):
        batches = [batches]
    with torch.cuda.device(dev):
        counts = torch.zeros(max(D * 4 * n_cells, 1), dtype=torch.int32, device=dev)
        hist = torch.zeros(2 * P, dtype=torch.int64, device=dev) if find else None
        seq = torch.zeros(2 * P * K * 4, dtype=torch.int64, device=dev) if find else None
        err = torch.zeros(1, dtype=torch.int64, device=dev)
        ends = torch.from_numpy(np.ascontiguousarray(lr.T.reshape(-1))).to(dev) if D else None
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        for b in batches:
            if b.n_records == 0:
                continue
            params = config.to_params(n_cells, max(int(b.max_read_extent()), 1))
            db = eng.upload(b)
            bc = db.as_c()
            rc = lib.mgatk_deletion_scan_device(
                eng.handle, ctypes.byref(params), ctypes.byref(bc), int(min_clip),
                ends.data_ptr() if D else None, ends.data_ptr() + 4 * D if D else None, D,
                counts.data_ptr(), hist.data_ptr() if find else None, seq.data_ptr() if find else None,
                err.data_ptr(), stream)
            if rc:
                eng._raise(rc)
            torch.cuda.synchronize(dev)              # the part's device buffers are released before the next upload
        torch.cuda.synchronize(dev)
        stats = np.zeros(8, np.uint64)
        stats[7] = np.uint64(err.cpu().numpy()[0])
        rc = lib.mgatk_check_stats(stats.ctypes.data)
        if rc:
            raise PileupKernelError(rc, lib.mgatk_status_string(rc).decode())
        c = counts.cpu().numpy().view(np.uint32)[: D * 4 * n_cells].reshape(D, 4, n_cells)
        h = hist.cpu().numpy().view(np.uint64).reshape(2, P) if find else None
        s = seq.cpu().numpy().view(np.uint64).reshape(2, P, K, 4) if find else None
    return DeletionScan(lr, c, h[0] if find else None, h[1] if find else None, s[0] if find else None,
                        s[1] if find else None, P, int(min_clip))


def _consensus(seq_p: np.ndarray) -> np.ndarray:
    """Argmax base (ties to the first of A, C, G, T) over the leading run of offsets with a nonzero total."""
    tot = seq_p.sum(axis=1)
    m = int(np.argmin(tot > 0)) if (tot == 0).any() else len(tot)
    return np.argmax(seq_p[:m], axis=1)


def _matches(codes: np.ndarray, starts: np.ndarray, c: np.ndarray, step: int) -> np.ndarray:
    """Starts s among `starts` with codes[s + step * j] == c[j] for every j (N, coded -1, never matches)."""
    ok = np.ones(len(starts), bool)
    for j, b in enumerate(c.tolist()):
        ok &= codes[starts + step * j] == b
    return starts[ok]


def find_deletions(scan: DeletionScan, reference, min_reads: int = 5, min_match: int = 10,
                   min_length: int = 100) -> np.ndarray:
    """Breakpoint pairs from the discovery histograms (DESIGN §8 "Deletions", pairing). `reference` is the run's
    reference allele per position (PileupResult.reference_alleles(), or a string). Returns CANDIDATES_DTYPE rows sorted
    by (l, r); `support` is 'both' when the pair is found from its left and its right candidate."""
    if scan.end_clip is None:
        raise ValueError("the scan ran without discovery (find=False)")
    if not 1 <= min_match <= DEL_KMER:
        raise ValueError(f"min_match must be in [1, {DEL_KMER}]")
    P = scan.mito_length
    ref = np.asarray(list(reference) if isinstance(reference, str) else reference)
    if len(ref) != P:
        raise ValueError(f"reference has {len(ref)} positions, the scan {P}")
    lut = {"A": 0, "C": 1, "G": 2, "T": 3}
    codes = np.array([lut.get(str(x).upper(), -1) for x in ref.tolist()], np.int64)
    min_gap = max(int(min_length), 1)
    left = np.nonzero(scan.end_clip >= min_reads)[0]
    right = np.nonzero(scan.start_clip >= min_reads)[0]
    found: dict = {}
    for l in left.tolist():
        c = _consensus(scan.end_seq[l])
        m = len(c)
        if m < min_match:
            continue
        starts = np.arange(l + 1 + min_gap, P - m + 1)            # r - l - 1 >= min_length, r + m - 1 < P
        hit = _matches(codes, starts, c, 1)
        if len(hit):
            pref = np.intersect1d(hit, right)
            found.setdefault((l, int(pref[0] if len(pref) else hit[0])), set()).add("left")
    for r in right.tolist():
        c = _consensus(scan.start_seq[r])
        m = len(c)
        if m < min_match:
            continue
        starts = np.arange(m - 1, r - min_gap)                     # r - l - 1 >= min_length, l - m + 1 >= 0
        hit = _matches(codes, starts, c, -1)
        if len(hit):
            pref = np.intersect1d(hit, left)
            found.setdefault((int(pref[-1] if len(pref) else hit[-1]), r), set()).add("right")
    out = np.zeros(len(found), CANDIDATES_DTYPE)
    letters = np.array(list("ACGT"))
    for k, (l, r) in enumerate(sorted(found)):
        sup = found[(l, r)]
        first, last = breakpoints_to_hgvs(l, r)
        out[k] = (l, r, deletion_name(l, r), first, last, r - l - 1, "both" if len(sup) == 2 else next(iter(sup)),
                  int(scan.end_clip[l]), int(scan.start_clip[r]), "".join(letters[_consensus(scan.end_seq[l])]),
                  "".join(letters[_consensus(scan.start_seq[r])]))
    return out


def deletion_heteroplasmy(scan: DeletionScan, deletions=None, cells=None) -> np.ndarray:
    """HETEROPLASMY_DTYPE rows, deletion-major then cell: the class counts of every selected cell (`cells`: a bool mask
    or column indices; None = all) for every deletion of the scan (or those of `deletions`, 1-based ranges), with
    heteroplasmy = del / (del + wt), del = clip_left + clip_right + gap, NaN when del + wt = 0."""
    n_cells = scan.counts.shape[2]
    if cells is None:
        idx = np.arange(n_cells)
    else:
        cells = np.asarray(cells)
        idx = np.nonzero(cells)[0] if cells.dtype == bool else cells.astype(np.int64)
    rows = {tuple(x): d for d, x in enumerate(scan.deletions.tolist())}
    if deletions is None:
        ds = list(range(len(scan.deletions)))
    else:
        want = [tuple(x) for x in breakpoints(deletions).tolist()]
        missing = [deletion_name(*w) for w in want if w not in rows]
        if missing:
            raise ValueError(f"not in the scan: {', '.join(missing)}")
        ds = [rows[w] for w in want]
    out = np.zeros(len(ds) * len(idx), HETEROPLASMY_DTYPE)
    for k, d in enumerate(ds):
        blk = out[k * len(idx): (k + 1) * len(idx)]
        c = scan.counts[d][:, idx].astype(np.int64)
        dl = c[0] + c[1] + c[2]
        tot = dl + c[3]
        blk["cell"] = idx
        blk["deletion"] = deletion_name(*scan.deletions[d])
        blk["index"] = d
        for j, name in enumerate(CLASSES):
            blk[name] = c[j]
        with np.errstate(invalid="ignore", divide="ignore"):
            blk["heteroplasmy"] = np.where(tot > 0, dl / np.where(tot > 0, tot, 1), np.nan)
    return out


def write_deletion_candidates(table: np.ndarray, path) -> None:
    """`deletion_candidates.tsv.gz`: a header line, one row per breakpoint pair, 1-based positions."""
    names = [n for n in CANDIDATES_DTYPE.names if n not in ("l", "r")]
    rows = ("\t".join(_fmt(row[n].item()) for n in names) + "\n" for row in table)
    _gzip_text(Path(path), ["\t".join(names) + "\n", *rows])


def read_deletion_candidates(path) -> np.ndarray:
    """A `deletion_candidates.tsv.gz` back as CANDIDATES_DTYPE."""
    with gzip.open(path, "rt") as f:
        header = f.readline().rstrip("\n").split("\t")
        body = [line.rstrip("\n").split("\t") for line in f]
    t = np.zeros(len(body), CANDIDATES_DTYPE)
    for j, name in enumerate(header):
        t[name] = [r[j] for r in body]
    t["l"], t["r"] = t["first"] - 2, t["last"]
    return t


def write_deletions(table: np.ndarray, barcodes, path) -> None:
    """`deletions.tsv.gz`: barcode, deletion, clip_left, clip_right, gap, wt, heteroplasmy for the rows of `table`
    (deletion_heteroplasmy) with del + wt > 0; `barcodes[cell]` names a cell; floats '.10g', NaN as NA."""
    names = ("barcode", "deletion", *CLASSES, "heteroplasmy")
    tot = sum(table[n].astype(np.int64) for n in CLASSES)
    lines = ["\t".join(names) + "\n"]
    for row in table[tot > 0].tolist():
        cell, name, _, cl, cr, gap, wt, het = row
        lines.append("\t".join([barcodes[cell], name, str(cl), str(cr), str(gap), str(wt), _fmt(het)]) + "\n")
    _gzip_text(Path(path), lines)


def read_deletions(path) -> list[dict]:
    """A `deletions.tsv.gz` back as dicts (counts int, heteroplasmy float, NA -> NaN)."""
    with gzip.open(path, "rt") as f:
        header = f.readline().rstrip("\n").split("\t")
        rows = [dict(zip(header, line.rstrip("\n").split("\t"))) for line in f]
    for r in rows:
        for n in CLASSES:
            r[n] = int(r[n])
        r["heteroplasmy"] = math.nan if r["heteroplasmy"] == "NA" else float(r["heteroplasmy"])
    return rows


def run_deletion_files(parts_of, res, config, barcode_list, out_dir, deletions=None, find: bool = False,
                       device: int = 0) -> np.ndarray | None:
    """The pipeline's deletion step: `parts_of()` yields the record parts the pileup saw (whitelist bc_idx), `res` its
    result (columns, alive cells, reference vote). Writes `deletions.tsv.gz` and, with `find`, `deletion_candidates.tsv.gz`
    into `out_dir`; returns the candidates (None without `find`)."""
    n_wl = len(barcode_list)
    cols = res.columns if res.columns is not None else np.arange(len(res.cell_qc))
    local_of = np.full(max(n_wl, 1), -1, np.int32)
    local_of[cols] = np.arange(len(cols), dtype=np.int32)
    n_cells = len(cols)

    def parts():
        for b in parts_of():
            ok = (b.bc_idx >= 0) & (b.bc_idx < n_wl)
            local = np.where(ok, local_of[np.clip(b.bc_idx, 0, len(local_of) - 1)], -1).astype(np.int32)
            yield ReadBatch(pos=b.pos, tlen=b.tlen, flag=b.flag, mapq=b.mapq, bc_idx=local, l_seq=b.l_seq,
                            n_cigar=b.n_cigar, blob_off=b.blob_off, blob=b.blob)

    given = breakpoints(deletions)
    scan = _scan(parts(), config, n_cells, given, find, device)
    cands = None
    if find:                                   # discovered pairs not given: counted in a second pass
        cands = find_deletions(scan, res.reference_alleles())
        known = {tuple(x) for x in given.tolist()}
        new = np.array([x for x in breakpoints(cands).tolist() if tuple(x) not in known], np.int32).reshape(-1, 2)
        for k in range(0, len(new), DEL_MAX):
            more = _scan(parts(), config, n_cells, new[k: k + DEL_MAX], False, device)
            scan = DeletionScan(np.concatenate([scan.deletions, more.deletions]),
                                np.concatenate([scan.counts, more.counts]), scan.end_clip, scan.start_clip,
                                scan.end_seq, scan.start_seq, scan.mito_length, scan.min_clip)
        write_deletion_candidates(cands, Path(out_dir) / "deletion_candidates.tsv.gz")
    table = deletion_heteroplasmy(scan, cells=res.alive())
    names = [barcode_list[int(c)] for c in cols]
    write_deletions(table, names, Path(out_dir) / "deletions.tsv.gz")
    return cands
