"""Time the clone step (DESIGN §8 "Clones"): mgatk_clone_knn_device, mgatk_clone_snn_device and mgatk_louvain_host.

For every (n, V) asked for, seeded clone-structured allele counts [V][3][n] are made on the GPU (40 clones, each with
its own set of variants at heteroplasmy 0.2-0.9, sampled coverage, 2 % noise; every row has a detected variant, so all
n cells are graph rows). The kNN call (the heteroplasmy pass and the fused all-pairs search with top-k) and the SNN call
are timed with CUDA events over --iters launches after a warm-up; the SNN graph build (numpy) and Louvain (host C++) with
a host clock. The rate is the pair-variant products n^2 V over the kNN time. The numpy oracle (oracle/clones.py rules)
is timed on the first --oracle-rows query rows against all n and scaled by n / rows; its lists are compared with the
GPU's. Prints one JSON line with the GPU's name and power limit read in the same run.

    python tools/bench_clones.py --rows 10000 100000 --variants 16 64 256 --out profiles/clones_bench.json
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


def make_counts(n: int, V: int, seed: int):
    """uint32 [V, 3, n] as an int32 tensor on cuda:0."""
    import torch
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(seed)
    n_clones = 40
    clone = torch.randint(0, n_clones, (n,), generator=g, device=dev)
    profile = torch.rand((n_clones, V), generator=g, device=dev, dtype=torch.float64) * 0.7 + 0.2
    profile *= torch.rand((n_clones, V), generator=g, device=dev) < max(0.1, 3.0 / V)
    het = profile[clone].t() * (0.7 + 0.6 * torch.rand((V, n), generator=g, device=dev, dtype=torch.float64))
    het += (torch.rand((V, n), generator=g, device=dev) < 0.02) * 0.1
    d = torch.randint(1, 60, (V, n), generator=g, device=dev, dtype=torch.int64)
    a = torch.minimum(torch.floor(het * d).to(torch.int64), d)
    own = (clone % V).unsqueeze(0)                                     # one detected variant per row at least
    a.scatter_(0, own, torch.maximum(a.gather(0, own), torch.ones_like(own)))
    f = a // 2
    return torch.stack([f, a - f, d], dim=1).to(torch.int32).contiguous()


def oracle_slice(x, rows: int, k: int):
    """(nbr, sim) of the first `rows` query rows by the oracle's rules, and the seconds it took."""
    import numpy as np
    t = time.perf_counter()
    n, V = x.shape
    acc = np.zeros((rows, n))
    for v in range(V):
        acc = acc + np.multiply.outer(x[:rows, v], x[:, v])
    self_dot = np.zeros(n)
    for v in range(V):
        self_dot = self_dot + x[:, v] * x[:, v]
    inv = 1.0 / np.sqrt(self_dot)
    cos = (acc * inv[:rows, None]) * inv[None, :]
    idx = np.arange(n)
    nbr = np.zeros((rows, k), np.int32)
    sim = np.zeros((rows, k))
    for i in range(rows):
        m = idx != i
        order = np.lexsort((idx[m], -cos[i, m]))[: k - 1]
        nbr[i, 0], sim[i, 0] = i, 1.0
        nbr[i, 1:], sim[i, 1:] = idx[m][order], cos[i, m][order]
    return nbr, sim, time.perf_counter() - t


def run(n: int, V: int, k: int, iters: int, warmup: int, oracle_rows: int) -> dict:
    import numpy as np
    import torch

    from mgatk2_b200.clones import louvain, snn_graph
    from mgatk2_b200.pileup import get_engine

    eng = get_engine(0)
    dev = torch.device("cuda", 0)
    counts = make_counts(n, V, seed=n + V)
    rows = torch.arange(n, dtype=torch.int32, device=dev)
    nbr = torch.empty((n, k), dtype=torch.int32, device=dev)
    sim = torch.empty((n, k), dtype=torch.float64, device=dev)
    w = torch.empty((n, k), dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(0)
    s = ctypes.c_void_p(stream.cuda_stream)
    lib, h = eng.lib, eng.handle

    def knn():
        rc = lib.mgatk_clone_knn_device(h, counts.data_ptr(), rows.data_ptr(), n, n, V, k, nbr.data_ptr(), sim.data_ptr(), s)
        assert rc == 0, lib.mgatk_last_error(h)

    def snn():
        rc = lib.mgatk_clone_snn_device(h, nbr.data_ptr(), n, k, w.data_ptr(), s)
        assert rc == 0, lib.mgatk_last_error(h)

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(stream)
        for _ in range(iters):
            fn()
        t1.record(stream)
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / iters

    knn_ms = timed(knn)
    snn_ms = timed(snn)
    nbr_h, sim_h, w_h = nbr.cpu().numpy(), sim.cpu().numpy(), w.cpu().numpy()
    t = time.perf_counter()
    csr = snn_graph(nbr_h, w_h)
    graph_s = time.perf_counter() - t
    t = time.perf_counter()
    labels, levels = louvain(*csr)
    louvain_s = time.perf_counter() - t

    c = counts.cpu().numpy().view(np.uint32).astype(np.uint64)
    a, d = (c[:, 0] + c[:, 1]).astype(np.float64), c[:, 2].astype(np.float64)
    x = np.ascontiguousarray(np.where(d > 0, a / np.maximum(d, 1.0), 0.0).T)
    r = min(oracle_rows, n)
    o_nbr, o_sim, o_s = oracle_slice(x, r, k)
    products = float(n) * n * V
    return {"n": n, "V": V, "k": k, "iters": iters, "knn_ms": round(knn_ms, 3), "snn_ms": round(snn_ms, 4),
            "snn_graph_s": round(graph_s, 3), "louvain_s": round(louvain_s, 3), "louvain_levels": levels,
            "n_clones_found": int(labels.max()), "snn_edges": int(len(csr[1])),
            "pair_variant_products": products, "products_per_s": round(products / (knn_ms * 1e-3), 1),
            "oracle_s_scaled": round(o_s * n / r, 2), "oracle_rows_timed": r,
            "oracle_slice_equal": bool(np.array_equal(o_nbr, nbr_h[:r]) and o_sim.tobytes() == sim_h[:r].tobytes())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, nargs="+", default=[10000, 100000])
    ap.add_argument("--variants", type=int, nargs="+", default=[16, 64, 256])
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--oracle-rows", type=int, default=64)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_clones.py needs a CUDA device")
    from mgatk2_b200.build import build_extension
    build_extension()
    line = dict(gpu_identity(), kernels="mgatk_clone_knn_device + mgatk_clone_snn_device, mgatk_louvain_host",
                runs=[run(n, v, a.k, a.iters, a.warmup, a.oracle_rows) for n in a.rows for v in a.variants])
    text = json.dumps(line)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
