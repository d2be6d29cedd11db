"""TEST INFRASTRUCTURE — plain numpy restatement of the variant sums (mgatk_variant_sums, DESIGN §8 "Variant
statistics"), not product code.

`oracle_variant_sums` works from exact uint32 counts [C, P, 4, 2] and coverage [C, P] (as `OracleResult` and
`PileupResult.counts()` / `.coverage()` give them), the reference allele of every position (0..3, -1 = N) and a cell
mask. Its output has the device's layout, so the same `mgatk2_b200.variants.finalize` turns both into floats.
"""
from __future__ import annotations

import numpy as np

from mgatk2_b200.variants import OVER_THRESHOLDS, VARIANT_SUMS_DTYPE, variant_mean


def reference_alleles(base_totals: np.ndarray) -> np.ndarray:
    """int [P]: first of A,C,G,T with the largest total, -1 when none is positive."""
    bt = np.asarray(base_totals, np.int64)
    ref = np.argmax(bt, axis=1).astype(np.int32)
    ref[bt.max(axis=1) <= 0] = -1
    return ref


def oracle_variant_sums(counts: np.ndarray, coverage: np.ndarray, ref: np.ndarray, mask: np.ndarray | None = None,
                        low_coverage_threshold: int = 10) -> np.ndarray:
    C, P = coverage.shape
    sel = np.ones(C, bool) if mask is None else np.asarray(mask, bool)
    cells = np.nonzero(sel)[0]
    L = int(low_coverage_threshold)
    out = np.zeros((P, 4), VARIANT_SUMS_DTYPE)
    ref = np.asarray(ref, np.int32)
    out["ref"] = ref[:, None]
    d_all = coverage[cells].astype(np.uint64)                                    # [N, P]
    for b in range(4):
        o = out[:, b]
        valid = (ref >= 0) & (ref != b)
        f = counts[cells, :, b, 0].astype(np.uint64)
        r = counts[cells, :, b, 1].astype(np.uint64)
        a = f + r
        d = d_all
        s = {}
        s["sum_fwd"], s["sum_rev"], s["sum_cov"] = f.sum(0), r.sum(0), d.sum(0)
        s["sum_ff"], s["sum_rr"], s["sum_fr"] = (f * f).sum(0), (r * r).sum(0), (f * r).sum(0)
        s["n_covered"] = (d > 0).sum(0)
        s["n_detected"] = s["n_strand"] = (a > 0).sum(0)
        s["n_conf_detected"] = ((f >= 2) & (r >= 2)).sum(0)
        s["n_low"] = (d < L).sum(0)
        over = np.stack([((d > 0) & (100 * a >= k * d)).sum(0) for k in OVER_THRESHOLDS], axis=1)
        # largest a / d over covered cells, cell by cell: a strictly larger cross product replaces, so ties keep the first
        best_a, best_d = np.zeros(P, np.uint64), np.zeros(P, np.uint64)
        for i in range(len(cells)):
            ai, di = a[i], d[i]
            better = (di > 0) & ((best_d == 0) | (ai * best_d > best_a * di))
            best_a = np.where(better, ai, best_a)
            best_d = np.where(better, di, best_d)
        mean = variant_mean(s["sum_fwd"], s["sum_rev"], s["sum_cov"])
        with np.errstate(divide="ignore", invalid="ignore"):
            u = np.where(d >= L, a.astype(np.float64) / d.astype(np.float64) - mean, 0.0)
        dev_sum, dev_sq = u.sum(0), (u * u).sum(0)
        for k, v in s.items():
            o[k] = np.where(valid, v, 0)
        o["n_over"] = np.where(valid[:, None], over, 0)
        o["max_alt"], o["max_cov"] = np.where(valid, best_a, 0), np.where(valid, best_d, 0)
        o["dev_sum"], o["dev_sq"] = np.where(valid, dev_sum, 0.0), np.where(valid, dev_sq, 0.0)
        o["valid"] = valid
        out[:, b] = o
    return out
