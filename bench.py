#!/usr/bin/env python
"""Benchmark of the per-cell chrM pileup hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (CUDA, C-ABI)
    python bench.py ... --dump-outputs DIR                       also write the last timed step's result to DIR/*.npy
    python bench.py --impl reference [...]                       the reference's own Python (baseline/_ref), C port beside it
    torchrun ... bench.py --gpus N --scaling strong              ONE configs[2]-shaped input split by barcode over N GPUs

A step is one pass of stages 1-6 over one batch of synthetic records. At N=1 the workload is
BASELINE.json configs[1] (2 000 cells x 20 M records, 2x50 bp, default `run` filters); at N>1 every
rank owns a barcode shard of that same size (weak scaling, no data-path collective). `value` is records/s
with inputs resident in HBM (CUDA events, max over ranks); `e2e` is the same metric through
`mgatk_pileup_host_submit` / `_wait` with pinned HOST buffers (H2D + kernels + D2H inside the timed region, two batches in
flight) next to a probe of the box's host -> device ceiling; `roofline` is the WHOLE step against the measured HBM
bandwidth, with the dominant kernel reported against its own algorithmic bytes; `cpu_baseline` is the unmodified
reference (kind "reference") on a bounded sample, with the C port on all host threads as `cpu_baseline.port`.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "dedup chrM reads/sec counted"
UNIT = "reads/s"
CONFIG_INDEX = 1
BASE_SEED = 20261018


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cells", type=int, default=2000)
    ap.add_argument("--records", type=int, default=20_000_000)
    ap.add_argument("--profile", default="atac50")
    ap.add_argument("--params", default="run", choices=["run", "tenx", "stress"],
                    help="filter set: run defaults (the bench line), tenx (configs[3]) or stress (configs[4]); "
                         "anything but `run` is a side measurement, not the bench line")
    ap.add_argument("--e2e-steps", type=int, default=None, help="timed steps of each e2e measurement (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed to DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verify", action="store_true", help="check per-cell QC rows against the oracle at full size")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak (the bench line): every rank owns a shard of --cells x --records. strong (side measurement): ONE "
                         "input of --strong-cells x --strong-records (BASELINE configs[2]) is split by barcode over the ranks")
    ap.add_argument("--strong-cells", type=int, default=10_000)
    ap.add_argument("--strong-records", type=int, default=200_000_000)
    ap.add_argument("--strong-parts", type=int, default=8, help="the strong-scaling input is the union of this many "
                    "barcode-disjoint parts (seeded per part, so it is the same input whatever the number of ranks)")
    a = ap.parse_args()
    if a.e2e_steps is None:
        a.e2e_steps = a.steps
    if a.steps < 1 or a.e2e_steps < 1:
        ap.error("--steps and --e2e-steps must be at least 1")
    return a


def config_dict(a, n_gpus):
    filt = {"run": "default run filters (q20 mapq30 d5 bias1.0, alignment_and_fragment_length dedup)",
            "tenx": "tenx filters (q0 mapq0 d5 alignment_start dedup)", "stress": "stress filters (q20 mapq30 d10 bias0.8)"}[a.params]
    if getattr(a, "scaling", "weak") == "strong":
        wl = (f"synthetic 10x-ATAC chrM, BASELINE configs[2] shape: ONE input of {a.strong_cells} cells x {a.strong_records} records "
              f"split by barcode over {n_gpus} GPU(s), profile {a.profile}, {filt}")
    else:
        wl = (f"synthetic 10x-ATAC chrM, BASELINE configs[{CONFIG_INDEX}]: {a.cells} cells x {a.records} records per GPU, "
              f"profile {a.profile}, {filt}")
    return {"workload": wl, "cells_per_gpu": a.cells, "records_per_gpu": a.records, "profile": a.profile,
            "sharding": f"by barcode, {n_gpus} shard(s), no data-path collective",
            "l2": "inputs per step (>2 GB) exceed the 126 MB L2; no explicit flush"}


def algorithmic_bytes(batch, n_cells, P=16569):
    """SURVEY §8(d): each input byte read once, each output byte written once.
    per record 15 + 4*n_cigar + ceil(L/2) + L; per (cell, position) 11 planes x 2 B; 32 B QC row per cell."""
    per_rec = 15 * batch.n_records + int((4 * batch.n_cigar.astype(np.int64) + (batch.l_seq.astype(np.int64) + 1) // 2
                                           + batch.l_seq).sum())
    return per_rec + n_cells * P * 22 + n_cells * 32


def default_params(n_cells, extent, which="run"):
    """ParamsC(min_baseq, min_mapq, min_distance_from_end, dedup_mode, max_strand_bias, min_reads_per_cell, P, ...)."""
    from mgatk2_b200._lib import ParamsC
    if which == "tenx":       # cli/options.py:172-236; min_distance_from_end stays 5 through the CLI (SURVEY Q1)
        return ParamsC(0, 0, 5, 1, 1.0, 0, 16569, n_cells, extent, 0)
    if which == "stress":     # BASELINE configs[4]: max-strand-bias 0.8, min-distance-from-end 10
        return ParamsC(20, 30, 10, 0, 0.8, 1, 16569, n_cells, extent, 0)
    return ParamsC(20, 30, 5, 0, 1.0, 1, 16569, n_cells, extent, 0)


# --------------------------------------------------------------------------- CPU arms
if __name__ == "__mp_main__" and os.environ.get("MGATK_REF_ACTIVATE"):
    # a spawned worker of the reference's own process pool (reference arm only): import the reference in its working order
    from baseline import ref_harness as _rh
    _rh._activate()


def cpu_sample(a, cells=None):
    """Bounded sample with the per-cell shape of the workload (same records per cell)."""
    from mgatk2_b200.synth import synth_batch
    cells = max(1, min(a.cells, 200 if cells is None else cells))
    recs = max(1000, int(a.records * cells / a.cells))
    return synth_batch(cells, recs, a.profile, seed=BASE_SEED + CONFIG_INDEX + 99), cells, recs


def filter_kwargs(which):
    return {"run": dict(min_baseq=20, min_mapq=30, min_distance_from_end=5, dedup_mode=0, max_strand_bias=1.0),
            "tenx": dict(min_baseq=0, min_mapq=0, min_distance_from_end=5, dedup_mode=1, max_strand_bias=1.0, min_reads_per_cell=0),
            "stress": dict(min_baseq=20, min_mapq=30, min_distance_from_end=10, dedup_mode=0, max_strand_bias=0.8)}[which]


def time_oracle(batch, cells, threads, steps, warmup, which="run"):
    from oracle.oracle import make_params, run_oracle
    p = make_params(cells, max_read_extent=batch.max_read_extent(), **filter_kwargs(which))
    for _ in range(warmup):
        run_oracle(batch, p, n_threads=threads)
    t0 = time.perf_counter()
    for _ in range(steps):
        run_oracle(batch, p, n_threads=threads)
    return (time.perf_counter() - t0) / steps


def port_figure(a, steps=3, warmup=1):
    """The C restatement (oracle/mgatk2_oracle.c) on all host threads: the CPU number the reference would reach if its
    Python loops were compiled. Reported next to the reference's own number, never instead of it."""
    threads = os.cpu_count() or 1
    sb, sc, sr = cpu_sample(a)
    dt = time_oracle(sb, sc, threads, steps, warmup, a.params)
    return {"value": sr / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{sc} cells x {sr} records per pass (same records/cell as the workload), oracle/mgatk2_oracle.c, "
                      f"{threads} threads over cells, mean of {steps} passes"}


def time_reference_python(a, steps, warmup, budget_s):
    """The reference's own Python (baseline/_ref, unmodified) through BAMReader + CellProcessor on a sample sized to
    `budget_s` seconds in total. Returns the cpu_baseline object (kind "reference") or None when it is not installed."""
    from baseline import ref_harness as rh
    if not rh.available():
        return None
    from mgatk2_b200.synth import make_whitelist
    kw = filter_kwargs(a.params)
    # calibration pass: one cell of the workload's depth
    cb, cc, cr = cpu_sample(a, cells=1)
    wl = make_whitelist(cc)
    path = rh.prepare(cb, wl)
    dt0, _, _, _ = rh.run_once(path, wl, **kw)
    rh.release(path)
    per_pass = budget_s / max(steps + warmup, 1)
    cells = int(max(1, min(a.cells, 64, per_pass / max(dt0, 1e-3))))
    sb, sc, sr = cpu_sample(a, cells=cells)
    wl = make_whitelist(sc)
    path = rh.prepare(sb, wl)                      # pysam-like read objects are built here, outside the clock
    try:
        for _ in range(warmup):
            rh.run_once(path, wl, **kw)
        tot, mode, stats = 0.0, "", {}
        for _ in range(steps):
            dt, stats, _, mode = rh.run_once(path, wl, **kw)
            tot += dt
    finally:
        rh.release(path)
    dt = tot / max(steps, 1)
    cores = 1 if mode.startswith("sequential") else (os.cpu_count() or 1)
    return {"value": sr / dt, "unit": UNIT, "cores": cores, "kind": "reference", "seconds_per_pass": dt,
            "sample": f"{sc} cells x {sr} records per pass (same records/cell as the workload); unmodified ollieeknight/mgatk2 "
                      f"from baseline/_ref: BAMReader.collect_reads_by_barcode + CellProcessor.process_cells_progressive, "
                      f"{mode}; pysam replaced by pre-decoded read objects (no BAM decoding inside the clock), "
                      f"{steps} timed passes after {warmup} warm-up",
            "reference_stats": {k: int(v) for k, v in stats.items() if isinstance(v, (int, np.integer))}}


def time_reference_pool(a, records_per_cell=3000):
    """Side figure of the reference arm: the reference's process pool at work. At the workload's depth the reference
    forces its sequential loop (`processors.py:99-101`), so its `--threads` never shows; this sample stays below 2 500
    reads per cell (one pass, all host cores, worker start-up included - the reference pays it on every run)."""
    from baseline import ref_harness as rh
    if not rh.available():
        return None
    from mgatk2_b200.synth import make_whitelist, synth_batch
    cores = os.cpu_count() or 1
    cells = int(min(256, 16 * cores))
    recs = cells * records_per_cell
    batch = synth_batch(cells, recs, a.profile, seed=BASE_SEED + CONFIG_INDEX + 199)
    wl = make_whitelist(cells)
    path = rh.prepare(batch, wl)
    try:
        dt, stats, _, mode = rh.run_once(path, wl, n_cores=cores, **filter_kwargs(a.params))
    finally:
        rh.release(path)
    return {"value": recs / dt, "unit": UNIT, "cores": cores, "kind": "reference", "seconds_per_pass": dt,
            "sample": f"{cells} cells x {recs} records ({records_per_cell} per cell: below the reference's 2500-reads-per-cell "
                      f"switch), one pass, {mode}"}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    port = port_figure(a)
    ref = time_reference_python(a, a.steps, a.warmup, budget_s=150.0)
    cpu = dict(ref, port=port) if ref else port
    try:
        pool = time_reference_pool(a)
        if pool:
            cpu["pool"] = pool
    except Exception as e:                                  # a side figure never fails the arm
        cpu["pool"] = {"unavailable": f"{type(e).__name__}: {e}"}
    v = cpu["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": cpu.get("seconds_per_pass", 0.0) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": config_dict(a, a.gpus),
        "cpu_baseline": cpu,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and clock-event reasons through NVML every few ms on a thread while the timed
    region runs (nvidia-smi -lms is too coarse for a region of tens of milliseconds)."""

    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index, period_s=0.004):
        import threading
        self.samples, self.bits, self.max_mhz, self.power = [], 0, None, []
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            import torch
            uuid = str(torch.cuda.get_device_properties(gpu_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            return

        def loop():
            nv = self.nv
            while not self._stop.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    self.bits |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                    self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
                except Exception:
                    pass
                self._stop.wait(period_s)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self._thread:
            self._stop.set()
            self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(k for k, b in self.REASONS.items() if self.bits & b),
                "samples": len(self.samples), "power_w_max": max(self.power) if self.power else None}


# --------------------------------------------------------------------------- outputs
DUMP_CELLS = 40          # planes of this many cells: 40 x 11 x 16569 float64 = 58 MB, the rest of a dump is below 1 MB
DUMP_LIMIT = 64 << 20


def dump_outputs(res, out_dir):
    """Write the PileupResult of a step (what a caller of the path receives) as .npy files of fixed shapes, so that two
    builds can be compared output for output on the same seeded input:
      planes.npy          float64 [DUMP_CELLS, 11, P]  exact planes (PLANE_NAMES order; entries saturated in the uint16
                                                       planes carry their value from the overflow list, as counts() / tn5()
                                                       / coverage() give them) of a fixed, seeded sample of cells;
                                                       planes_cells.npy (float64) lists the sampled rows
      cell_qc_<f>.npy     float64 [n_cells]            every field of the per-cell QC rows
      base_totals.npy     float64 [P, 4]
      stats.npy           float64 [8]                  STATS_FIELDS order
    Every value is an integer below 2**53, so the float64 copies are exact."""
    from mgatk2_b200._lib import N_PLANES
    from mgatk2_b200.engine import STATS_FIELDS
    n_cells = len(res.planes)
    rows = np.sort(np.random.default_rng(BASE_SEED).choice(n_cells, min(n_cells, DUMP_CELLS), replace=False))
    arrays = {"planes": np.stack([res.plane(k)[rows] for k in range(N_PLANES)], axis=1).astype(np.float64),
              "planes_cells": rows.astype(np.float64),
              **{f"cell_qc_{f}": res.cell_qc[f].astype(np.float64) for f in res.cell_qc.dtype.names},
              "base_totals": res.base_totals.astype(np.float64),
              "stats": np.array([res.stats[k] for k in STATS_FIELDS], np.float64)}
    total = sum(v.nbytes for v in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT})")
    os.makedirs(out_dir, exist_ok=True)
    for name, v in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), v)


# --------------------------------------------------------------------------- our arm
def run_b200(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the pileup path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from mgatk2_b200.build import build_extension
    if rank == 0:
        build_extension()
    if world > 1:
        dist.barrier()
    from mgatk2_b200.engine import PileupEngine
    from mgatk2_b200.synth import synth_batch

    t_gen = time.perf_counter()
    if a.scaling == "strong":
        # one input, split by barcode: the union of `strong_parts` barcode-disjoint parts; rank r counts parts
        # r*parts/world .. (r+1)*parts/world - 1 merged back into coordinate order (what routing one BAM by barcode gives)
        if a.strong_parts % world or a.strong_cells % a.strong_parts or a.strong_records % a.strong_parts:
            raise SystemExit("--strong-parts must divide --strong-cells and --strong-records and be a multiple of the ranks")
        from mgatk2_b200.batch import ReadBatch as _RB
        per, cpp = a.strong_parts // world, a.strong_cells // a.strong_parts
        parts = []
        for k in range(per):
            m = rank * per + k
            b = synth_batch(cpp, a.strong_records // a.strong_parts, a.profile, seed=BASE_SEED + 7000 + m)
            b.bc_idx = np.where(b.bc_idx >= 0, b.bc_idx + k * cpp, b.bc_idx).astype(np.int32)
            parts.append(b)
        batch = _RB.concat(parts)
        if per > 1:
            batch = batch.take(np.argsort(batch.pos, kind="stable"))
        del parts
        a.cells, a.records = cpp * per, batch.n_records
    else:
        batch = synth_batch(a.cells, a.records, a.profile, seed=BASE_SEED + CONFIG_INDEX + 1000 * rank)
    t_gen = time.perf_counter() - t_gen
    extent = batch.max_read_extent()
    params = default_params(a.cells, extent, a.params)
    eng = PileupEngine(local)

    # pinned host staging (e2e) and device-resident copy (value)
    from mgatk2_b200.batch import FIELDS, ReadBatch
    pinned = {}
    for name, _ in FIELDS:
        src = torch.from_numpy(getattr(batch, name))
        pinned[name] = torch.empty_like(src, pin_memory=True).copy_(src)
    pbatch = ReadBatch(**{name: pinned[name].numpy() for name, _ in FIELDS})
    dbatch = eng.upload(pbatch, pinned_src=pinned)
    dout = eng.alloc_device_outputs(a.cells, 16569, batch.n_records, max_read_extent=extent)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up, then K timed steps with inputs resident in HBM ----
    for _ in range(max(a.warmup, 3)):
        eng.run_device(dbatch, params, dout)
    barrier()
    clocks = ClockSampler(local)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps):
        eng.run_device(dbatch, params, dout)
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    last = eng.download(dout, params) if a.dump_outputs and rank == 0 else None     # outputs of the last timed step
    launches = eng.launch_count() * a.steps
    # per-stage device times (events inside the library, same stream), averaged over K more steps
    stage_acc = {}
    for _ in range(a.steps):
        eng.run_device(dbatch, params, dout)
        torch.cuda.synchronize()
        for k, v in eng.stage_times().items():
            stage_acc[k] = stage_acc.get(k, 0.0) + v / a.steps
    clock_info = clocks.stop()
    res = eng.download(dout, params)           # also checks the device error bits

    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / a.steps
    total_records = a.records * world
    value = total_records / (ms_step * 1e-3)
    if a.scaling == "strong":          # the one cross-cell quantity of the path: base totals of all shards, one NCCL all-reduce
        tot = torch.from_numpy(res.base_totals.copy()).cuda()
        kept_all = torch.tensor([res.stats["filtered_reads"]], dtype=torch.int64, device="cuda")
        if world > 1:
            dist.all_reduce(tot)
            dist.all_reduce(kept_all)
        strong_check = {"filtered_reads_all_ranks": int(kept_all.item()), "base_totals_sum_all_ranks": int(tot.sum().item())}

    # ---- e2e: host buffers through the C ABI, every step uploads its inputs and downloads its result ----
    # (1) blocking call per step (mgatk_pileup_host); (2) the same steps through submit / wait with two batches in
    #     flight, which is how a caller with more than one batch drives the library (upload k+1 next to download k).
    # the box's host -> device ceiling with all ranks copying at once (plain pinned cudaMemcpyAsync, 1 GiB x 8): what the
    # upload of e2e competes for
    probe_src = torch.empty(1 << 30, dtype=torch.uint8, pin_memory=True)
    probe_dst = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    probe_dst.copy_(probe_src, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(8):
        probe_dst.copy_(probe_src, non_blocking=True)
    torch.cuda.synchronize()
    dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    h2d_ceiling_gbs = 8 * (1 << 30) * world / float(dt.item()) / 1e9
    del probe_src, probe_dst
    hout = eng.alloc_host_outputs(a.cells, 16569)
    hout2 = eng.alloc_host_outputs(a.cells, 16569)
    eng.run_host(pbatch, params, out=hout)      # warm-up: device buffers get allocated here
    for _, r in eng.run_host_many([pbatch] * 2, lambda b: params, [hout, hout2]):
        pass
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        r_e2e = eng.run_host(pbatch, params, out=hout)
    torch.cuda.synchronize()
    dt = torch.tensor([(time.perf_counter() - t0) / a.e2e_steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_blocking = total_records / float(dt.item())
    barrier()
    t0 = time.perf_counter()
    for _, r in eng.run_host_many([pbatch] * a.e2e_steps, lambda b: params, [hout, hout2]):
        assert r.stats["filtered_reads"] == res.stats["filtered_reads"]
    torch.cuda.synchronize()
    dt = torch.tensor([(time.perf_counter() - t0) / a.e2e_steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    e2e_value = total_records / float(dt.item())
    h2d = pbatch.nbytes()
    d2h = int(hout["planes"].nbytes + hout["cell_qc"].nbytes + hout["stats"].nbytes + hout["base_totals"].nbytes)
    assert r_e2e.stats["filtered_reads"] == res.stats["filtered_reads"]

    if a.verify:
        from oracle.oracle import make_params, run_oracle
        ora = run_oracle(batch, make_params(a.cells, params.min_baseq, params.min_mapq, params.min_distance_from_end,
                                            params.dedup_mode, params.max_strand_bias, params.min_reads_per_cell,
                                            max_read_extent=extent), n_threads=os.cpu_count() or 1, dense=False)
        for f in ("n_reads", "n_paired", "sum_depth", "covered", "max_depth", "median_lo", "median_hi"):
            np.testing.assert_array_equal(res.cell_qc[f], ora.cell_qc[f])
        np.testing.assert_array_equal(res.base_totals, ora.base_totals)
        assert all(res.stats[k] == ora.stats[k] for k in ("filtered_reads", "dup_with_length", "dup_position_only"))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if a.dump_outputs:
        dump_outputs(last, a.dump_outputs)

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # Whole-step roofline (BASELINE.md §4): every input byte read once + every output byte written once, over the time of
    # stages 1-6. The dominant kernel is reported next to it against ITS OWN algorithmic bytes (what that launch must
    # read and write given its place in the pipeline), never against the whole job's.
    bytes_alg = algorithmic_bytes(batch, a.cells)
    slot_bytes = 32 if extent <= 56 else (16 + 16 * min(8, max(2, (extent + 31) // 32)) + 31) // 32 * 32
    in_bytes = bytes_alg - a.cells * 16569 * 22 - a.cells * 32
    out_bytes = a.cells * 16569 * 22 + a.cells * 32
    stage1, kept = int(res.stats["stage1_reads"]), int(res.stats["filtered_reads"])
    stage_bytes = {"filter+planes+partition": in_bytes + 6 * batch.n_records + stage1 * slot_bytes,   # + the histogram pass
                   "dedup": stage1 * slot_bytes + kept * slot_bytes,
                   "pileup": kept * slot_bytes + out_bytes,
                   "totals+median": a.cells * 16569 * 2}
    dom = max(stage_acc, key=stage_acc.get) if stage_acc else "pileup"
    dom_ms = stage_acc.get(dom, ms_step)
    dom_bytes = stage_bytes.get(dom, bytes_alg)
    traffic, dom_traffic, traffic_src = None, None, None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get("step_dram_bytes"), tj.get("source")
        dom_traffic = (tj.get("stages") or {}).get(dom)
    achieved = bytes_alg / (ms_step * 1e-3) / 1e9
    roofline = {"bound": "hbm", "scope": "whole step (stages 1-6, all kernels)", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_bytes_per_step": bytes_alg, "step_ms": ms_step,
                "dominant_kernel": {"stage": dom, "ms": dom_ms, "algorithmic_bytes_per_launch": dom_bytes,
                                    "achieved": dom_bytes / (dom_ms * 1e-3) / 1e9,
                                    "frac": dom_bytes / (dom_ms * 1e-3) / 1e9 / peak, "traffic": dom_traffic},
                "stage_ms": stage_acc, "stage_algorithmic_bytes": stage_bytes}

    cpu = None
    if not a.no_cpu_baseline:
        port = port_figure(a)
        ref = time_reference_python(a, steps=1, warmup=0, budget_s=20.0)
        cpu = dict(ref, port=port) if ref else port

    print(json.dumps({
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None, "dtype": "u32",
        "data": "synthetic", "config": config_dict(a, world), "clocks": clock_info,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": a.e2e_steps,
                "mode": "mgatk_pileup_host_submit/_wait, two batches in flight, pinned host buffers",
                "blocking_value": e2e_blocking,
                "h2d_gbs": h2d * world * e2e_value / total_records / 1e9,
                "h2d_ceiling_gbs": h2d_ceiling_gbs,
                "h2d_ceiling_note": "plain pinned 1 GiB host->device copies on all ranks at once; the upload of e2e cannot beat it"},
        "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        "counted": {"total_reads": res.stats["total_reads"], "filtered_reads": res.stats["filtered_reads"],
                    "dup_with_length": res.stats["dup_with_length"], "sum_depth": int(res.cell_qc["sum_depth"].sum())},
        "synth_seconds": t_gen, **({"strong": strong_check} if a.scaling == "strong" else {}),
        **({"verified": "per-cell QC rows (reads, pairs, depth sum, covered, max, both medians), base totals and the "
                        "three counters equal to the oracle at full size"} if a.verify else {}),
    }))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)
