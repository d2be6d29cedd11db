"""`MtDNAPipeline` — the caller of the three-call seam (reference src/core/pipeline.py:23-181), so a BAM file goes
in and the reference's text outputs come out with the counting on the GPU:

    BAMReader.collect_reads_by_barcode()  ->  CellProcessor.process_cells_progressive()  ->  writer.finalize()

Same constructor keywords, same return value of `run()`, same files (`output/output.{A,C,G,T,coverage}.txt.gz`,
`output/output.depthTable.txt`, `output/<mito>_refAllele.txt`, `qc/cell_stats.csv`, `qc/summary.txt`), or with
`output_format="hdf5"` the reference's default `output/counts.h5` + `output/metadata.h5` (written by `h5lite`; the HTML
report that follows them in the reference is out of scope).
No BAM index is required (the native reader scans without one; the reference would call `pysam.index`)."""
from __future__ import annotations

import datetime
import logging
import time
from pathlib import Path

from .barcodes import load_barcodes
from .config import PipelineConfig
from .exceptions import InvalidInputError

logger = logging.getLogger(__name__)
VERSION = "mgatk2_b200 round 1"


def write_run_summary(run_metadata: dict, output_path: Path):
    """`qc/summary.txt` in the layout of file_io/formats.py:49-57: title, rule, `key: value` lines, then the indented
    `parameters` block when there is one."""
    params = run_metadata.get("parameters")
    lines = ["mgatk2 Run Summary", "=" * 20]
    lines += [f"{k}: {v}" for k, v in run_metadata.items() if k != "parameters"]
    if "parameters" in run_metadata:
        lines += ["", "Parameters:"] + [f"  {k}: {v}" for k, v in params.items()]
    Path(output_path).write_text("\n".join(lines) + "\n")


class MtDNAPipeline:
    def __init__(self, bam_path: str, barcodes: list, output_dir, config: PipelineConfig | None = None,
                 output_format: str = "standard", barcode_metadata=None, sample_name: str = "mgatk2",
                 report_title: str | None = None, report_subtitle: str | None = None, working_directory: str | None = None,
                 device: int = 0, devices: list | None = None, max_batch_records: int | None = None,
                 call_variants: bool = False, find_clones: bool = False, clone_markers: bool = False,
                 deletions: list | None = None, find_deletions: bool = False):
        """`call_variants=True` adds `output/variant_stats.tsv.gz` and `output/variant_cells.tsv.gz` (variants.py) after
        the reference's outputs, which stay as they are. `find_clones=True` implies it and adds `output/clones.tsv.gz` and
        `output/clone_variants.tsv.gz` (clones.py, the called variants, default parameters). `clone_markers=True` implies
        `find_clones` and adds `output/clone_markers.tsv.gz` (markers.py: each clone against the other graph cells).
        `deletions` (1-based HGVS ranges (first, last)) and `find_deletions=True` add one more pass over the same records
        (deletions.py): `output/deletions.tsv.gz` per cell and deletion, and with `find_deletions` the breakpoint pairs
        found from soft clips in `output/deletion_candidates.tsv.gz`, which are counted too."""
        self.bam_path = Path(bam_path)
        self.barcodes = set(barcodes)
        self.barcode_list = list(barcodes)
        self.output_dir = Path(output_dir)
        self.config = config or PipelineConfig()
        self.output_format = output_format.lower()
        self.barcode_metadata = barcode_metadata
        self.sample_name = sample_name
        self.devices = list(devices) if devices else [device]      # GPUs of this box; the cells are split between them
        self.device = self.devices[0]
        self.max_batch_records = max_batch_records                  # larger contigs are streamed in parts (dispatch.py)
        self.clone_markers = bool(clone_markers)
        self.find_clones = bool(find_clones) or self.clone_markers
        self.call_variants = bool(call_variants) or self.find_clones
        self.deletions = None if deletions is None else [(int(f), int(t)) for f, t in deletions]
        self.find_deletions = bool(find_deletions)
        if not self.bam_path.exists():
            raise InvalidInputError(f"BAM file not found: {bam_path}")
        from .bamio import BamFile, pick_mito_contig
        with BamFile(str(self.bam_path)) as bam:                          # pipeline.py:62-76
            if self.config.mito_chr not in bam.references:
                alt = pick_mito_contig(bam.references)
                if alt is None:
                    raise InvalidInputError(f"Mitochondrial chromosome '{self.config.mito_chr}' not found. "
                                            f"Available: {', '.join(bam.references[:10])}")
                logger.warning("Using '%s' instead of '%s'", alt, self.config.mito_chr)
                self.config.mito_chr = alt
        self.output_dir.mkdir(parents=True, exist_ok=True)

    def run(self) -> dict:
        from .processors import CellProcessor
        from .readers import BAMReader
        from .writers import DenseHDF5Writer, DenseTextWriter
        start = time.time()
        logger.info("Collecting reads from BAM by barcode...")
        reader = BAMReader(str(self.bam_path), self.config, self.barcodes, barcode_list=self.barcode_list,
                           devices=self.devices, max_batch_records=self.max_batch_records)
        reads_by_barcode, stats = reader.collect_reads_by_barcode()
        if not reads_by_barcode:
            logger.error("No reads found for any barcodes!")
            return {}
        n_cells_input = len(reads_by_barcode)
        t_write = time.time()
        if self.output_format == "hdf5":                                  # pipeline.py:88-94, the default of `mgatk2 run`
            writer = DenseHDF5Writer(self.output_dir, self.config, self.barcode_list, barcode_metadata=self.barcode_metadata)
        else:
            writer = DenseTextWriter(self.output_dir, self.config, self.barcode_list)
        cell_results = CellProcessor(self.config, self.output_dir).process_cells_progressive(reads_by_barcode, writer)
        if not cell_results:
            logger.error("No cells passed quality filters")
            return {}
        qc_dir = self.output_dir / "qc"
        writer.finalize(qc_dir)
        if self.call_variants:
            from .pileup import get_engine
            from .variants import _Source, write_variant_files
            src = _Source(reads_by_barcode.result, get_engine(self.device))         # one upload for every file below
            called, counts = write_variant_files(src, self.barcode_list, self.output_dir / "output")
            logger.info("%d variants called", len(called))
            if self.find_clones:
                from .clones import write_clone_files
                clones = write_clone_files(src, self.barcode_list, self.output_dir / "output", called, counts)
                logger.info("%d clones", clones.n_clones)
                if self.clone_markers:
                    from .markers import clone_markers, write_clone_markers
                    write_clone_markers(clone_markers(src, clones, counts=counts),
                                        self.output_dir / "output" / "clone_markers.tsv.gz")
        if self.deletions is not None or self.find_deletions:
            from .deletions import run_deletion_files
            t_del = time.time()
            one = getattr(reader, "batch", None)             # a one-batch input is still in memory; a stream is re-read
            parts_of = (lambda: iter([one])) if one is not None else reader._parts
            cands = run_deletion_files(parts_of, reads_by_barcode.result, self.config, self.barcode_list,
                                       self.output_dir / "output", deletions=self.deletions, find=self.find_deletions,
                                       device=self.device)
            reader.timings["deletions_s"] = time.time() - t_del
            logger.info("deletions: %d given, %s found", len(self.deletions or []),
                        "-" if cands is None else len(cands))
        self.timings = dict(getattr(reader, "timings", {}), write_s=time.time() - t_write, total_s=time.time() - start)
        c = self.config
        write_run_summary({                                               # analysis/qc.py:68-93
            "mgatk_version": VERSION, "run_date": datetime.datetime.now().isoformat(), "input_bam": str(self.bam_path),
            "output_dir": str(self.output_dir), "reference": c.mito_chr, "reference_length": c.mito_length,
            "cells_total": n_cells_input, "cells_passed_qc": len(cell_results),
            "cells_failed_qc": n_cells_input - len(cell_results),
            "parameters": {"min_base_quality": c.quality.min_baseq, "min_mapping_quality": c.quality.min_mapq,
                           "min_reads_per_cell": c.min_reads_per_cell, "max_strand_bias": c.quality.max_strand_bias,
                           "skip_deduplication": c.dedup.skip, "use_fragment_length_dedup": c.dedup.use_fragment_length,
                           "barcode_tag": c.barcode_tag, "mito_chr": c.mito_chr, "n_cores": c.performance.n_cores},
        }, qc_dir / "summary.txt")
        logger.info("Pipeline complete")
        logger.info("Elapsed time: %ds", int(time.time() - start))
        self.stats = stats
        return {"cells_processed": n_cells_input, "cells_passed_qc": len(cell_results),
                "mean_reads": sum(r["n_reads"] for r in cell_results) / len(cell_results) if cell_results else 0}


def run_pipeline(bam_path: str, output_dir: str, barcode_file: str | None = None, min_barcode_reads: int = 10,
                 barcode_tag: str = "CB", mito_chr: str = "chrM", output_format: str = "standard", device: int = 0,
                 devices: list | None = None, max_batch_records: int | None = None, call_variants: bool = False,
                 find_clones: bool = False, clone_markers: bool = False, deletions: list | None = None,
                 find_deletions: bool = False, **config_kwargs) -> dict:
    """core.pipeline.run_pipeline (pipeline.py:184-270): whitelist from file / singlecell.csv / the BAM itself, then
    `MtDNAPipeline.run()` (`call_variants`, `find_clones`, `clone_markers`, `deletions`, `find_deletions`: as there). `config_kwargs` are `PipelineConfig` keywords (min_baseq, min_mapq, max_strand_bias,
    skip_deduplication, use_fragment_length_dedup, min_reads_per_cell, ...)."""
    barcodes, metadata = load_barcodes(barcode_file, bam_path, barcode_tag=barcode_tag, mito_chr=mito_chr,
                                       min_barcode_reads=min_barcode_reads)
    config = PipelineConfig(barcode_tag=barcode_tag, mito_chr=mito_chr, **config_kwargs)
    return MtDNAPipeline(bam_path, barcodes, Path(output_dir), config, output_format=output_format,
                         barcode_metadata=metadata, device=device, devices=devices,
                         max_batch_records=max_batch_records, call_variants=call_variants,
                         find_clones=find_clones, clone_markers=clone_markers, deletions=deletions,
                         find_deletions=find_deletions).run()
