"""Time the deletion scan (DESIGN §8 "Deletions"): mgatk_deletion_scan_device and the pipeline's extra pass.

1. The scan on a resident batch: seeded synth_batch inputs (C2: 2 000 cells x 20 M records of 2x50 bp; stress150: 2 000
   cells x --stress-records records of 2x150 bp with soft clips and indels), run filters, 1 / 16 / 256 seeded deletions
   (lengths 500-8 000), with and without discovery. CUDA events over --iters calls after two warm-ups; the algorithmic
   bytes are the 17 bytes per record of the SoA arrays the relevance pass reads (pos, tlen, flag, mapq, bc_idx, l_seq)
   plus the blobs of the records whose CIGAR is read.
2. The pipeline's extra wall time: run_pipeline on a BAM written by bamio, with and without deletions (16 given +
   find_deletions), as one batch and streamed in four parts; a host clock around each run after one warm-up run.
3. The plain-Python oracle (oracle/deletions.py) on the first --oracle-records records of C2, scaled by n / that.
Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/bench_deletions.py --out profiles/deletions_bench.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import shutil
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.bench_variants import gpu_identity  # noqa: E402


def seeded_deletions(n: int, P: int = 16569, seed: int = 7):
    import numpy as np
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        first = int(rng.integers(200, P - 8200))
        out.append((first, first + int(rng.integers(500, 8000))))
    return out


def time_scan(eng, batch, config, n_cells, dels, find, iters):
    import numpy as np
    import torch
    from mgatk2_b200.deletions import DEL_KMER, breakpoints
    dev = torch.device("cuda", eng.device)
    lr = breakpoints(dels)
    D, P = len(lr), int(config.mito_length)
    db = eng.upload(batch)
    params = config.to_params(n_cells, max(int(batch.max_read_extent()), 1))
    counts = torch.zeros(max(D * 4 * n_cells, 1), dtype=torch.int32, device=dev)
    hist = torch.zeros(2 * P, dtype=torch.int64, device=dev)
    seq = torch.zeros(2 * P * DEL_KMER * 4, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int64, device=dev)
    ends = torch.from_numpy(np.ascontiguousarray(lr.T.reshape(-1))).to(dev)
    stream = torch.cuda.current_stream(dev)
    bc = db.as_c()

    def call():
        rc = eng.lib.mgatk_deletion_scan_device(eng.handle, ctypes.byref(params), ctypes.byref(bc), 5, ends.data_ptr(),
                                                ends.data_ptr() + 4 * D, D, counts.data_ptr(),
                                                hist.data_ptr() if find else None, seq.data_ptr() if find else None,
                                                err.data_ptr(), ctypes.c_void_p(stream.cuda_stream))
        assert rc == 0, eng.lib.mgatk_last_error(eng.handle)

    for _ in range(2):
        call()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        call()
    e1.record(stream)
    torch.cuda.synchronize(dev)
    assert int(err.cpu()[0]) == 0
    return e0.elapsed_time(e1) / iters


def walked_bytes(batch, dels, find):
    """Blob bytes of the stage-1 records whose CIGAR the relevance pass reads (start within the extent of a breakpoint,
    or every one with discovery) — the 16-byte units that hold their CIGAR and, for counted ones, SEQ."""
    import numpy as np
    from mgatk2_b200.deletions import breakpoints
    st1 = ((batch.flag & 0x904) == 0) & (batch.bc_idx >= 0)
    if find:
        walk = st1
    else:
        E = batch.max_read_extent()
        bps = np.sort(breakpoints(dels).reshape(-1))
        k = np.searchsorted(bps, batch.pos)
        walk = st1 & (k < len(bps)) & (bps[np.minimum(k, len(bps) - 1)] <= batch.pos.astype(np.int64) + E - 1)
    return int(16 * ((4 * batch.n_cigar[walk].astype(np.int64) + 15) // 16).sum())


def pipeline_extra(n_cells, n_records, iters_dir):
    from mgatk2_b200 import run_pipeline
    from mgatk2_b200.bamio import write_bam
    from mgatk2_b200.synth import make_whitelist, synth_batch
    batch = synth_batch(n_cells, n_records, "stress150", seed=424242)
    wl = make_whitelist(n_cells, seed=5)
    bam = os.path.join(iters_dir, "in.bam")
    write_bam(bam, batch, wl, write_index=False)
    dels = seeded_deletions(16)
    out = {}
    for name, mbr in (("one_batch", None), ("streamed_4_parts", n_records // 4 + 1)):
        times = {}
        for label, kw in (("warmup", {}), ("without", {}), ("with", dict(deletions=dels, find_deletions=True))):
            d = os.path.join(iters_dir, f"{name}_{label}")
            t = time.perf_counter()
            run_pipeline(bam, d, min_barcode_reads=1, max_batch_records=mbr, **kw)
            times[label] = time.perf_counter() - t
            shutil.rmtree(d)
        out[name] = {"without_s": round(times["without"], 3), "with_s": round(times["with"], 3),
                     "extra_s": round(times["with"] - times["without"], 3)}
    out["records"], out["cells"] = int(batch.n_records), n_cells
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--records", type=int, default=20_000_000)
    ap.add_argument("--stress-records", type=int, default=10_000_000)
    ap.add_argument("--cells", type=int, default=2000)
    ap.add_argument("--deletions", type=int, nargs="+", default=[1, 16, 256])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--oracle-records", type=int, default=20000)
    ap.add_argument("--pipeline-records", type=int, default=1_000_000)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from mgatk2_b200.config import PipelineConfig
    from mgatk2_b200.pileup import get_engine
    from mgatk2_b200.synth import synth_batch
    from oracle import deletions as od
    eng = get_engine(0)
    config = PipelineConfig()
    line = {"tool": "bench_deletions", **gpu_identity(), "iters": a.iters, "scan": {}}
    for shape, profile, n in (("C2", "atac50", a.records), ("stress150", "stress150", a.stress_records)):
        t = time.perf_counter()
        batch = synth_batch(a.cells, n, profile, seed=20261022)
        gen_s = time.perf_counter() - t
        rows = []
        for D in a.deletions:
            dels = seeded_deletions(D)
            for find in (False, True):
                ms = time_scan(eng, batch, config, a.cells, dels, find, a.iters)
                soa = 17 * batch.n_records
                blob = walked_bytes(batch, dels, find)
                rows.append({"deletions": D, "discovery": find, "ms": round(ms, 4),
                             "soa_plus_cigar_GB_per_s": round((soa + blob) / ms / 1e6, 1)})
                print(shape, rows[-1], flush=True)
        line["scan"][shape] = {"records": int(batch.n_records), "cells": a.cells, "synth_s": round(gen_s, 1), "rows": rows}
        if shape == "C2":
            sl = batch.slice(0, a.oracle_records)
            t = time.perf_counter()
            od.scan(sl, a.cells, 16569, [(l - 2, r) for l, r in seeded_deletions(16)], find=True)
            dt = time.perf_counter() - t
            line["oracle_C2_16_deletions_discovery_s"] = round(dt * batch.n_records / sl.n_records, 1)
        del batch
    with tempfile.TemporaryDirectory() as d:
        line["pipeline"] = pipeline_extra(500, a.pipeline_records, d)
    text = json.dumps(line)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
