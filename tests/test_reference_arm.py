"""The reference arm of bench.py (baseline/ref_harness.py) runs the UNMODIFIED reference installed into baseline/_ref:
its counters must equal the oracle's, so the CPU number printed next to the GPU one is a number of the real code path.
tests/golden/reference_arm_counters.json keeps what the unmodified reference counted on two seeded samples of the bench
workload; the oracle must reproduce those counters on every checkout. Where the reference is installed it is also run
here, on a small batch, against the oracle."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from baseline import ref_harness as rh  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_arm_counters.json")


def test_reference_counters_equal_the_oracle():
    from mgatk2_b200.synth import make_whitelist, synth_batch
    from oracle.oracle import make_params, run_oracle
    for s in json.load(open(GOLDEN))["samples"]:
        batch = synth_batch(s["cells"], s["records"], s["profile"], seed=s["seed"])
        ora = run_oracle(batch, make_params(s["cells"], max_read_extent=batch.max_read_extent(), **s["params"]),
                         n_threads=4, dense=False)
        ref = s["reference_stats"]
        assert ref["total_reads"] == ora.stats["total_reads"] == batch.n_records
        assert ref["filtered_reads"] == ora.stats["filtered_reads"]
        assert ref["duplicate_reads_with_length"] == ora.stats["dup_with_length"]
        assert ref["duplicate_reads_position_only"] == ora.stats["dup_position_only"]
        assert ref["n_barcodes"] == int((ora.cell_qc["n_reads"] > 0).sum())
    if not rh.available():
        return
    cells = 2                                            # above 2500 reads per cell: the reference takes its sequential loop
    batch = synth_batch(cells, 14000, "atac50", seed=11)
    wl = make_whitelist(cells)
    path = rh.prepare(batch, wl)
    try:
        dt, stats, n_cells, mode = rh.run_once(path, wl, n_cores=1)
    finally:
        rh.release(path)
    ora = run_oracle(batch, make_params(cells, max_read_extent=batch.max_read_extent()), n_threads=2)
    assert dt > 0 and n_cells <= cells
    assert stats["total_reads"] == ora.stats["total_reads"] == batch.n_records
    assert stats["filtered_reads"] == ora.stats["filtered_reads"]
    assert stats["duplicate_reads_with_length"] == ora.stats["dup_with_length"]
    assert stats["duplicate_reads_position_only"] == ora.stats["dup_position_only"]
    assert n_cells == int((ora.cell_qc["n_reads"] > 0).sum())           # cells the reference hands to its writer
    assert mode.startswith("sequential")
