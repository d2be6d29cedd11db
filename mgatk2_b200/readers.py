"""`BAMReader` — the first call of the drop-in seam (reference src/processing/readers.py:22-201).

Same constructor and `collect_reads_by_barcode() -> (reads_by_barcode, stats)` contract. The reference
materialises one `SimpleRead` per kept record; here the records stay in a structure-of-arrays batch and
stages 1-6 run on the GPU inside this call (dedup cannot be separated from the device pipeline).
`reads_by_barcode` is a read-only mapping barcode -> `CellReads` whose `len()` is the number of kept
reads, iterated in first-seen (BAM) order like the reference's dict; `CellProcessor` consumes it.
"""
from __future__ import annotations

import logging
from collections.abc import Mapping
from pathlib import Path

import numpy as np

from .batch import ReadBatch
from .engine import PileupResult
from .exceptions import BAMReadError
from .pileup import get_engine

logger = logging.getLogger(__name__)


class CellReads:
    """Stand-in for the reference's per-barcode list of reads: sized, and carries the device result."""

    __slots__ = ("barcode", "index", "n_reads", "result")

    def __init__(self, barcode: str, index: int, n_reads: int, result: PileupResult):
        self.barcode, self.index, self.n_reads, self.result = barcode, index, n_reads, result

    def __len__(self):
        return self.n_reads

    def __bool__(self):
        return self.n_reads > 0


class ReadsByBarcode(Mapping):
    """barcode -> CellReads in first-seen (BAM) order. `order` holds rows of the result; with compacted columns
    (`result.columns`) row k belongs to whitelist entry `columns[k]`."""

    def __init__(self, barcode_list: list[str], order: np.ndarray, result: PileupResult):
        self.result = result
        cols = result.columns
        name = (lambda c: barcode_list[int(cols[c])]) if cols is not None else (lambda c: barcode_list[c])
        self._cells = {name(c): CellReads(name(c), int(c), int(result.cell_qc["n_reads"][c]), result) for c in order.tolist()}

    def __getitem__(self, k):
        return self._cells[k]

    def __iter__(self):
        return iter(self._cells)

    def __len__(self):
        return len(self._cells)

    def pop(self, k, *default):          # the reference's processors pop cells as they go (processors.py:70,125)
        return self._cells.pop(k, *default)


def whitelist_index(barcode_list: list[str]) -> dict[str, int]:
    """Barcode -> column. Duplicated whitelist entries: the last index wins (writers.py:41)."""
    return {bc: i for i, bc in enumerate(barcode_list)}


class BAMReader:
    def __init__(self, bam_path: str, config, barcodes, *, barcode_list: list[str] | None = None,
                 batch: ReadBatch | None = None, device: int = 0, devices: list | None = None,
                 max_batch_records: int | None = None):
        """`barcodes` is the set the reference passes (pipeline.py:80); `barcode_list` (pipeline.barcode_list)
        fixes the column order. `batch` supplies already-decoded records (tests, synthetic data); without it
        the BAM at `bam_path` is decoded by `mgatk2_b200.bamio`. `devices` lists the GPUs of this box to count on
        (cells are split between them, `dispatch.py`); `max_batch_records` is the largest batch counted in one go -
        a contig with more records is streamed in parts through device-resident planes."""
        from .dispatch import DEFAULT_MAX_BATCH_RECORDS
        self.bam_path = Path(bam_path)
        self.config = config
        self.barcodes = barcodes
        self.barcode_list = list(barcode_list) if barcode_list is not None else sorted(barcodes)
        self.devices = list(devices) if devices else [device]
        self.device = self.devices[0]
        self.max_batch_records = int(max_batch_records or DEFAULT_MAX_BATCH_RECORDS)
        self._batch = batch
        if batch is None:
            if not self.bam_path.exists():
                raise BAMReadError(str(bam_path), "File does not exist")
            self._validate_bam_file()

    def _validate_bam_file(self):
        """readers.py:35-61: the file opens as a BAM, a mitochondrial contig is in the header (config.mito_chr is
        updated to the name found), and one of the first 1001 chrM records carries the barcode tag."""
        from .bamio import BamFile, pick_mito_contig
        from .exceptions import NoBarcodeTagsError, NoChrMReadsError
        with BamFile(str(self.bam_path)) as bam:
            mito = pick_mito_contig(bam.references)
            if mito is None:
                raise NoChrMReadsError(str(self.bam_path), bam.references)
            if self.config.mito_chr != mito:
                logger.info("Using mitochondrial chromosome: %s", mito)
                self.config.mito_chr = mito
            head, _, _ = bam.fetch(mito, self.config.barcode_tag, threads=1, max_records=1001)
        if head.n_records > 1000 and not (head.bc_idx != -1).any():
            raise NoBarcodeTagsError(str(self.bam_path), self.config.barcode_tag, 1000)

    def _parts(self):
        """The contig's records as an iterator of batches cut on reference_start borders, each at most about
        `max_batch_records` long (one batch for everything that fits)."""
        if self._batch is not None:
            b = self._batch
            if not b.is_sorted():
                raise ValueError("records are not sorted by reference_start")
            n_parts = -(-b.n_records // self.max_batch_records)
            yield from (b.split_on_start_borders(n_parts) if n_parts > 1 else [b])
            return
        from .bamio import iter_bam_chrM          # native BGZF/BAM decoder (csrc/bamio.cpp), SURVEY §8 f-1
        yield from iter_bam_chrM(str(self.bam_path), self.config, whitelist_index(self.barcode_list), self.max_batch_records)

    def _count_barcodes(self) -> np.ndarray:
        """Records per whitelist entry on the contig: one extra pass over the file, only for streamed inputs whose
        whitelist is too long to give every entry a column."""
        counts = np.zeros(max(len(self.barcode_list), 1), np.int64)
        for b in self._parts():
            ok = (b.bc_idx >= 0) & (b.bc_idx < len(self.barcode_list))
            counts += np.bincount(b.bc_idx[ok], minlength=len(counts))
        return counts

    def collect_reads_by_barcode(self):
        import itertools
        import time

        from . import dispatch
        self.timings = {}                       # seconds per phase of the last call (tools/bench_pipeline.py)
        n_wl = len(self.barcode_list)
        try:
            t0 = time.perf_counter()
            parts = self._parts()
            first = next(parts, None)
            second = next(parts, None) if first is not None else None
            self.timings["ingest_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            if first is None:
                first = ReadBatch.from_records([])
            if second is None:                  # everything fits one batch: exact overflow list, no accumulation
                batch = first
                if not batch.is_sorted():
                    raise ValueError("records are not sorted by reference_start")
                res = dispatch.run_one_batch(batch, self.config, n_wl, self.devices)
                ok = ((batch.flag & 0x904) == 0) & dispatch.usable(batch, n_wl)
                cells, first_idx = np.unique(batch.bc_idx[ok], return_index=True)
                first_seen = np.full(max(n_wl, 1), np.iinfo(np.int64).max, np.int64)
                first_seen[cells] = first_idx
                self.streamed = False
                self.batch = batch              # the one batch, for a later pass over the same records (deletions.py)
            else:
                counts = None
                plane_bytes = 11 * 2 * ((int(self.config.mito_length) + 63) // 64 * 64)
                if n_wl * plane_bytes > dispatch.MAX_STREAM_PLANE_BYTES * len(self.devices):
                    counts = self._count_barcodes()
                first_seen = np.full(max(n_wl, 1), np.iinfo(np.int64).max, np.int64)
                res = dispatch.run_stream(itertools.chain([first, second], parts), self.config, n_wl, self.devices,
                                          records_per_barcode=counts, first_seen=first_seen)
                self.streamed = True
                self.batch = None
            self.timings["gpu_host_abi_s"] = time.perf_counter() - t0
            if res.stats["n_empty_seq"]:
                raise ValueError("record without SEQ passed the filters")       # readers.py:157 raises here
        except BAMReadError:
            raise
        except Exception as e:
            raise BAMReadError(str(self.bam_path), f"Read error: {e}") from e

        # first-seen order of barcodes with kept reads: a barcode's first stage-1 record is never a duplicate
        cols = res.columns if res.columns is not None else np.arange(n_wl)
        order = np.argsort(first_seen[cols], kind="stable") if len(cols) else np.zeros(0, np.int64)
        order = order[first_seen[cols][order] < np.iinfo(np.int64).max]
        order = order[res.cell_qc["n_reads"][order] > 0]
        reads_by_barcode = ReadsByBarcode(self.barcode_list, order, res)

        st = res.stats
        if not self.config.dedup.skip and st["total_reads"]:                      # readers.py:170-180
            removed = st["dup_with_length"] if self.config.dedup.use_fragment_length else st["dup_position_only"]
            logger.info("%d duplicate reads removed (%.1f%%)", removed, removed / st["total_reads"] * 100)
        logger.info("Kept %s reads from %s barcodes", f"{st['filtered_reads']:,}", f"{len(reads_by_barcode):,}")
        stats = {"total_reads": st["total_reads"], "filtered_reads": st["filtered_reads"],
                 "n_barcodes": len(reads_by_barcode),
                 "duplicate_reads_with_length": st["dup_with_length"],
                 "duplicate_reads_position_only": st["dup_position_only"]}
        return reads_by_barcode, stats
