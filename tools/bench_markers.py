"""Time the clone-marker ranks (DESIGN §8 "Clone markers"): mgatk_marker_ranks_device.

For every (C, V, detection rate) asked for, seeded counts [V][3][C] are made on the GPU: coverage 1-59, a detected cell
(at the given rate) has 1..d alternate reads, so x = a / d takes few distinct values and ties are common, as in real
data; labels 1..G (G = 40) cover every cell, so all C cells are the population. The call is timed with CUDA events over
--iters launches after a warm-up. A variant with more than kMarkerS (4 096) nonzero x takes the merge fallback: at 50 %
detection and 100 000 cells every variant does. The scipy oracle (`scipy.stats.mannwhitneyu`, asymptotic with
continuity correction, one call per (variant, group) as R's per-feature `wilcox.test`) is timed on the first
--oracle-variants variants and scaled by V / that; its p values are compared with the GPU's through `markers.wilcoxon`.
Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/bench_markers.py --cells 10000 100000 --variants 16 64 256 1024 --out profiles/markers_bench.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_variants import gpu_identity  # noqa: E402

S = 4096                                            # kMarkerS


def make_inputs(C: int, V: int, G: int, rate: float, seed: int):
    """(counts int32 [V, 3, C] holding uint32 values, labels int32 [C]) on cuda:0."""
    import torch
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(seed)
    d = torch.randint(1, 60, (V, C), generator=g, device=dev, dtype=torch.int64)
    hit = torch.rand((V, C), generator=g, device=dev) < rate
    a = torch.where(hit, 1 + (torch.rand((V, C), generator=g, device=dev) * d).long().clamp(max=d - 1), 0)
    f = a // 2
    counts = torch.stack([f, a - f, d], dim=1).to(torch.int32).contiguous()
    labels = torch.randint(1, G + 1, (C,), generator=g, device=dev, dtype=torch.int32)
    return counts, labels


def run(C: int, V: int, G: int, rate: float, iters: int, warmup: int, oracle_variants: int) -> dict:
    import numpy as np
    import scipy.stats as ss
    import torch

    from mgatk2_b200.markers import wilcoxon
    from mgatk2_b200.pileup import get_engine

    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    counts, labels = make_inputs(C, V, G, rate, seed=C + V + int(rate * 100))
    rank2 = torch.empty(V * G, dtype=torch.int64, device=dev)
    ties = torch.empty(V, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(0)
    s = ctypes.c_void_p(stream.cuda_stream)
    lib, h = eng.lib, eng.handle

    def call():
        rc = lib.mgatk_marker_ranks_device(h, counts.data_ptr(), labels.data_ptr(), C, V, G, rank2.data_ptr(),
                                           ties.data_ptr(), s)
        assert rc == 0, lib.mgatk_last_error(h)

    for _ in range(warmup):
        call()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(iters):
        call()
    t1.record(stream)
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / iters

    c = counts.cpu().numpy().view(np.uint32).astype(np.uint64)
    a, d = (c[:, 0] + c[:, 1]).astype(np.float64), c[:, 2].astype(np.float64)
    x = np.where(d > 0, a / np.maximum(d, 1.0), 0.0)
    lab = labels.cpu().numpy()
    r2 = rank2.cpu().numpy().view(np.uint64).reshape(V, G)
    tie = ties.cpu().numpy().view(np.uint64)
    nnz = (x > 0).sum(axis=1)
    k = min(oracle_variants, V)
    worst = 0.0
    t = time.perf_counter()
    for v in range(k):
        for grp in range(1, G + 1):
            m = lab == grp
            want = ss.mannwhitneyu(x[v, m], x[v, ~m], alternative="two-sided", method="asymptotic",
                                   use_continuity=True).pvalue
            got = wilcoxon(r2[v, grp - 1], tie[v], int(m.sum()), C)[3]
            worst = max(worst, abs(got - want) / want if want > 0 else abs(got - want))
    o_s = time.perf_counter() - t
    return {"C": C, "V": V, "G": G, "detection": rate, "iters": iters, "ms": round(ms, 4),
            "cells_per_s": round(C * V / (ms * 1e-3), 1), "nnz_mean": round(float(nnz.mean()), 1),
            "variants_fallback": int((nnz > S).sum()), "oracle_s_scaled": round(o_s * V / k, 2),
            "oracle_variants_timed": k, "oracle_p_max_rel_diff": worst}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, nargs="+", default=[10000, 100000])
    ap.add_argument("--variants", type=int, nargs="+", default=[16, 64, 256, 1024])
    ap.add_argument("--rates", type=float, nargs="+", default=[0.05, 0.5])
    ap.add_argument("--groups", type=int, default=40)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--oracle-variants", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_markers.py needs a CUDA device")
    from mgatk2_b200.build import build_extension
    build_extension()
    line = dict(gpu_identity(), kernels="mgatk_marker_ranks_device (k_marker_split + k_marker_rank)",
                runs=[run(c, v, a.groups, r, a.iters, a.warmup, a.oracle_variants)
                      for c in a.cells for r in a.rates for v in a.variants])
    text = json.dumps(line)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
