"""mgatk2_b200 — B200-native per-cell chrM pileup hot path of ollieeknight/mgatk2.

The package mirrors the reference's seam (`BAMReader`, `CellProcessor`, `process_barcode_worker`,
`PileupGenerator`, `PipelineConfig`) over hand-written sm_100a kernels behind a C ABI
(include/mgatk2_b200.h). Importing the package does not need a GPU; constructing a `PileupEngine` does.
"""
from .batch import ReadBatch
from .config import DeduplicationConfig, PerformanceConfig, PipelineConfig, QualityThresholds
from .exceptions import (BAMReadError, InvalidInputError, MgatkError, NoBarcodeTagsError, PileupKernelError,
                         ProcessingError)

__all__ = ["ReadBatch", "PipelineConfig", "QualityThresholds", "DeduplicationConfig", "PerformanceConfig",
           "MgatkError", "InvalidInputError", "ProcessingError", "BAMReadError", "NoBarcodeTagsError",
           "PileupKernelError", "BAMReader", "CellProcessor", "process_barcode_worker", "PileupGenerator",
           "PileupEngine", "MtDNAPipeline", "run_pipeline", "load_singlecell_csv", "extract_barcodes_from_bam",
           "DenseTextWriter", "DenseHDF5Writer", "report_inputs",
           "VARIANT_SUMS_DTYPE", "variant_sums", "finalize", "call_variants", "variant_cells",
           "allele_frequencies", "find_clones", "clone_variants", "find_markers", "clone_markers",
           "scan_deletions", "find_deletions", "deletion_heteroplasmy"]


def __getattr__(name):        # heavy pieces (ctypes library, torch) load on first use
    if name == "BAMReader":
        from .readers import BAMReader
        return BAMReader
    if name in ("CellProcessor", "process_barcode_worker"):
        from . import processors
        return getattr(processors, name)
    if name == "PileupGenerator":
        from .pileup import PileupGenerator
        return PileupGenerator
    if name in ("MtDNAPipeline", "run_pipeline"):
        from . import pipeline
        return getattr(pipeline, name)
    if name in ("load_singlecell_csv", "extract_barcodes_from_bam"):
        from . import barcodes
        return getattr(barcodes, name)
    if name in ("DenseTextWriter", "DenseHDF5Writer"):
        from . import writers
        return getattr(writers, name)
    if name == "report_inputs":
        from .report import report_inputs
        return report_inputs
    if name in ("VARIANT_SUMS_DTYPE", "variant_sums", "finalize", "call_variants", "variant_cells"):
        from . import variants
        return getattr(variants, name)
    if name in ("allele_frequencies", "find_clones", "clone_variants"):
        from . import clones
        return getattr(clones, name)
    if name in ("find_markers", "clone_markers"):
        from . import markers
        return getattr(markers, name)
    if name in ("scan_deletions", "find_deletions", "deletion_heteroplasmy"):
        from . import deletions
        return getattr(deletions, name)
    if name == "PileupEngine":
        from .engine import PileupEngine
        return PileupEngine
    raise AttributeError(name)
