"""Time mgatk_variant_stats_device on resident planes (DESIGN §8 "Variant statistics").

Planes of seeded small counts are made on the GPU for every cell count asked for (2 000 and 10 000 cells of chrM are
0.73 GB and 3.6 GB of planes, both larger than the 126 MB L2), with the base totals of those planes and an empty
overflow list. The call is timed with CUDA events over --iters warm launches. The algorithmic bytes are 14 B per
(cell, position) and pass (three alt letters on both strands and coverage, uint16) and the kernel makes two passes;
the numpy oracle (oracle/variants.py) is timed on the same planes, downloaded, over the first --oracle-positions
positions and scaled to the contig. Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/bench_variants.py --cells 2000 10000 --out profiles/variants_bench.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def gpu_identity() -> dict:
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out["power_limit"], out["max_sm_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:          # the numbers are still worth printing without it
        out["power_limit"] = f"unknown ({e})"
    return out


def run(n_cells: int, P: int, iters: int, warmup: int, oracle_positions: int) -> dict:
    import numpy as np
    import torch

    from mgatk2_b200._lib import OutputsC, ParamsC
    from mgatk2_b200.engine import pos_pad
    from mgatk2_b200.pileup import get_engine
    from mgatk2_b200.variants import VARIANT_SUMS_DTYPE
    from oracle.variants import oracle_variant_sums, reference_alleles

    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    ppad = pos_pad(P)
    g = torch.Generator(device=dev).manual_seed(n_cells)
    planes = torch.zeros((n_cells, 11, ppad), dtype=torch.int32, device=dev)
    planes[:, :8, :P] = torch.randint(0, 4, (n_cells, 8, P), generator=g, device=dev, dtype=torch.int32)
    planes[:, 0, :P] += torch.randint(0, 40, (n_cells, P), generator=g, device=dev, dtype=torch.int32)   # reference-like A
    planes[:, 10] = planes[:, :8].sum(1)
    totals = planes[:, :8, :P].to(torch.int64).sum(0).view(4, 2, P).sum(1).t().contiguous()
    planes = planes.to(torch.uint16)
    stats = torch.zeros(8, dtype=torch.int64, device=dev)
    out = torch.empty(P * 4 * VARIANT_SUMS_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    params = ParamsC()
    params.n_cells, params.mito_length = n_cells, P
    oc = OutputsC(planes.data_ptr(), None, stats.data_ptr(), totals.data_ptr(), None, 0)
    stream = torch.cuda.current_stream(0)

    def launch():
        rc = eng.lib.mgatk_variant_stats_device(eng.handle, ctypes.byref(params), ctypes.byref(oc), None, 10, out.data_ptr(),
                                                ctypes.c_void_p(stream.cuda_stream))
        assert rc == 0, eng.lib.mgatk_last_error(eng.handle)

    for _ in range(warmup):
        launch()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record(stream)
    for _ in range(iters):
        launch()
    t1.record(stream)
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / iters
    gpu_sums = out.cpu().numpy().view(VARIANT_SUMS_DTYPE).reshape(P, 4)

    # numpy oracle on the same planes (first oracle_positions positions, scaled to P)
    k = min(oracle_positions, P)
    host = planes[:, :, :k].cpu().numpy().astype(np.uint32)
    counts = np.stack([host[:, j] for j in range(8)], axis=-1).reshape(n_cells, k, 4, 2)
    ref = reference_alleles(totals.cpu().numpy())
    t = time.perf_counter()
    ora = oracle_variant_sums(counts, host[:, 10], ref[:k])
    oracle_s = (time.perf_counter() - t) * P / k
    same = all(np.array_equal(ora[f], gpu_sums[:k][f]) for f in VARIANT_SUMS_DTYPE.names if f not in ("dev_sum", "dev_sq"))
    bytes_per_pass = 14 * n_cells * P
    return {"n_cells": n_cells, "mito_length": P, "ms": round(ms, 4), "iters": iters,
            "algorithmic_bytes_per_pass": bytes_per_pass, "passes": 2,
            "achieved_GBps_two_passes": round(2 * bytes_per_pass / (ms * 1e-3) / 1e9, 1),
            "plane_bytes": int(planes.numel() * 2),
            "oracle_s_scaled": round(oracle_s, 3), "oracle_positions_timed": k, "oracle_integer_fields_equal": bool(same)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cells", type=int, nargs="+", default=[2000, 10000])
    ap.add_argument("--mito-length", type=int, default=16569)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--oracle-positions", type=int, default=2048)
    ap.add_argument("--out", default=None, help="also append the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_variants.py needs a CUDA device")
    from mgatk2_b200.build import build_extension
    build_extension()
    line = dict(gpu_identity(), kernel="mgatk_variant_stats_device",
                runs=[run(c, a.mito_length, a.iters, a.warmup, a.oracle_positions) for c in a.cells])
    text = json.dumps(line)
    print(text)
    if a.out:
        with open(a.out, "a") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
