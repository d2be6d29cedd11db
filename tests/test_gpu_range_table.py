"""k_pileup_main reads each chunk's candidate reads from a per-unit table of 518 entries (chrM's chunks of 32 positions).
A unit that spans more chunks - a sparse cell on a longer contig - finds its ranges by search instead. These batches mix
dense cells (units of a few hundred chunks, table) with sparse ones (one unit across the whole contig, search) on
contigs just above and well above the table's size, and check both entry points against the oracle."""
from __future__ import annotations

import numpy as np
import pytest

from mgatk2_b200.synth import synth_batch
from tests.test_gpu_shapes import engine, run_both_entries, sorted_concat  # noqa: F401  (engine: module fixture)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("profile", ["atac50", "stress150"])
@pytest.mark.parametrize("P", [16577, 40000])
def test_units_wider_than_the_range_table(engine, P, profile):  # noqa: F811
    n_dense, n_sparse = 16, 16
    dense = synth_batch(n_dense, 40_000, profile, seed=31 + P % 89, mito_length=P)
    sparse = synth_batch(n_sparse, 400, profile, seed=37 + P % 83, mito_length=P)
    sparse.bc_idx = np.where(sparse.bc_idx >= 0, sparse.bc_idx + n_dense, sparse.bc_idx).astype(np.int32)
    batch = sorted_concat([dense, sparse])
    n_cells = n_dense + n_sparse
    host, dev, ora = run_both_entries(engine, batch, n_cells, mito_length=P)
    assert ora.coverage.shape == (n_cells, P)
    assert ora.coverage[n_dense:].sum() > 0 and ora.coverage[:n_dense].sum() > 0
