"""TEST INFRASTRUCTURE — plain numpy / Python restatement of the clone step (DESIGN §8 "Clones"), not product code.

Every float operation is an IEEE fp64 add, multiply, square root or divide in the order DESIGN §8 states: numpy's
elementwise ufuncs round each operation and never fuse a multiply with an add, so the similarities, the SNN weights and
the Louvain labels are those of the device and of `mgatk_louvain_host`, bit for bit.
"""
from __future__ import annotations

import numpy as np


def allele_frequencies(counts: np.ndarray) -> np.ndarray:
    """fp64 [V, C]: x = (f + r) / d, 0 where d = 0, from uint32 counts [V, 3, C]."""
    c = np.asarray(counts, np.uint64)
    a, d = (c[:, 0] + c[:, 1]).astype(np.float64), c[:, 2].astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(d > 0, a / np.where(d > 0, d, 1.0), 0.0)


def graph_rows(x: np.ndarray, mask: np.ndarray | None = None) -> np.ndarray:
    """int32: the selected cells with x > 0 for at least one variant, ascending."""
    hit = (x > 0).any(axis=0) if len(x) else np.zeros(x.shape[1], bool)
    if mask is not None:
        hit &= np.asarray(mask, bool)
    return np.nonzero(hit)[0].astype(np.int32)


def dots(xr: np.ndarray, block: int = 512) -> np.ndarray:
    """fp64 [n, n]: dot(i, j) = sum over v ascending of acc = acc + x[i, v] * x[j, v], from 0."""
    n, V = xr.shape
    out = np.zeros((n, n))
    for i0 in range(0, n, block):
        acc = np.zeros((min(block, n - i0), n))
        for v in range(V):
            acc = acc + np.multiply.outer(xr[i0:i0 + block, v], xr[:, v])
        out[i0:i0 + block] = acc
    return out


def knn(xr: np.ndarray, k: int):
    """(nbr int32 [n, k_eff], sim fp64 [n, k_eff]) of the rows xr [n, V]: i itself with 1.0, then the k_eff - 1 other
    rows with the largest cos(i, j) = (dot(i, j) * inv[i]) * inv[j], ties to the lower row; inv[i] = 0 for an all-zero
    row."""
    n = len(xr)
    k_eff = min(k, n)
    dd = dots(xr)
    self_dot = np.diag(dd).copy()
    with np.errstate(divide="ignore"):
        inv = np.where(self_dot > 0, 1.0 / np.sqrt(self_dot), 0.0)      # an all-zero row: every cosine 0
    cos = (dd * inv[:, None]) * inv[None, :]
    nbr = np.zeros((n, k_eff), np.int32)
    sim = np.zeros((n, k_eff))
    idx = np.arange(n)
    for i in range(n):
        others = idx != i
        j, s = idx[others], cos[i, others]
        order = np.lexsort((j, -s))[: k_eff - 1]                # cos descending, then row ascending
        nbr[i, 0], sim[i, 0] = i, 1.0
        nbr[i, 1:], sim[i, 1:] = j[order], s[order]
    return nbr, sim


def snn_weights(nbr: np.ndarray) -> np.ndarray:
    """fp64 [n, k_eff]: s / (2 k_eff - s), s = |N(i) ∩ N(nbr[i, t])|."""
    n, k = nbr.shape
    sets = [set(r.tolist()) for r in nbr]
    w = np.zeros((n, k))
    for i in range(n):
        for t in range(k):
            s = len(sets[i] & sets[int(nbr[i, t])])
            w[i, t] = float(s) / float(2 * k - s)
    return w


def snn_graph(nbr: np.ndarray, w: np.ndarray, prune: float = 1.0 / 15):
    """Symmetric CSR (indptr int64, indices int32, weights fp64) of the kNN pairs with w >= prune, diagonal included."""
    n = len(nbr)
    edges = {}
    for i in range(n):
        for t in range(nbr.shape[1]):
            j, wt = int(nbr[i, t]), float(w[i, t])
            edges[(i, j)] = wt
            edges[(j, i)] = wt
    keys = sorted(e for e, wt in edges.items() if not wt < prune)
    indptr = np.zeros(n + 1, np.int64)
    for i, _ in keys:
        indptr[i + 1] += 1
    return (np.cumsum(indptr).astype(np.int64), np.array([j for _, j in keys], np.int32),
            np.array([edges[e] for e in keys], np.float64))


def _phase1(indptr, indices, weights, resolution, comm):
    n = len(indptr) - 1
    k = []
    m2 = 0.0
    for i in range(n):
        s = 0.0
        for e in range(indptr[i], indptr[i + 1]):
            s = s + weights[e]
        k.append(s)
        m2 = m2 + s
    tot = [0.0] * n
    for i in range(n):
        tot[comm[i]] = tot[comm[i]] + k[i]
    if not m2 > 0.0:
        return False
    any_move = False
    for _ in range(100):
        moved = False
        for i in range(n):
            old = comm[i]
            tot_old = tot[old]
            tot[old] = tot_old - k[i]
            wc = {old: 0.0}
            for e in range(indptr[i], indptr[i + 1]):
                j = indices[e]
                if j == i:
                    continue
                c = comm[j]
                wc[c] = wc.get(c, 0.0) + weights[e]

            def gain(c):
                return wc[c] - ((resolution * (tot[c] * k[i])) / m2)
            own = gain(old)
            best, best_gain = old, own
            for c in wc:
                g = gain(c)
                if g > best_gain or (g == best_gain and c < best):
                    best, best_gain = c, g
            if best != old and best_gain > own:
                comm[i] = best
                tot[best] = tot[best] + k[i]
                moved = True
            else:
                tot[old] = tot_old
        if not moved:
            break
        any_move = True
    return any_move


def louvain(indptr, indices, weights, resolution: float = 1.0):
    """(labels int32 [n] in 1..K, levels) by the rules of DESIGN §8 "Clones"."""
    indptr = [int(v) for v in indptr]
    indices = [int(v) for v in indices]
    weights = [float(v) for v in weights]
    n0 = len(indptr) - 1
    node_of = list(range(n0))
    levels = 0
    while True:
        n = len(indptr) - 1
        comm = list(range(n))
        if not _phase1(indptr, indices, weights, resolution, comm):
            break
        levels += 1
        first = {}
        for i in range(n):
            first.setdefault(comm[i], i)
        ids = {c: r for r, c in enumerate(sorted(first, key=first.get))}
        node_of = [ids[comm[v]] for v in node_of]
        agg = {}
        for i in range(n):                                   # (i asc, j asc): the order each sum is taken in
            for e in range(indptr[i], indptr[i + 1]):
                key = (ids[comm[i]], ids[comm[indices[e]]])
                agg[key] = agg.get(key, 0.0) + weights[e]
        keys = sorted(agg)
        nc = len(ids)
        cnt = [0] * (nc + 1)
        for c, _ in keys:
            cnt[c + 1] += 1
        indptr = list(np.cumsum(cnt).tolist())
        indices = [d for _, d in keys]
        weights = [agg[e] for e in keys]
    n = len(indptr) - 1
    size = [0] * n
    first = [-1] * n
    for i, c in enumerate(node_of):
        size[c] += 1
        if first[c] < 0:
            first[c] = i
    order = sorted(range(n), key=lambda c: (-size[c], first[c]))
    number = [0] * n
    for r, c in enumerate(order):
        number[c] = r + 1
    return np.array([number[c] for c in node_of], np.int32), levels


def oracle_find_clones(counts: np.ndarray, mask: np.ndarray | None = None, k: int = 10, resolution: float = 1.0,
                       prune: float = 1.0 / 15):
    """labels int32 [C] (0 = NA or not selected) and the pieces: rows, nbr, sim, snn weights, CSR."""
    x = allele_frequencies(counts)
    rows = graph_rows(x, mask)
    labels = np.zeros(x.shape[1], np.int32)
    if len(rows) == 0:
        return labels, dict(rows=rows)
    nbr, sim = knn(np.ascontiguousarray(x[:, rows].T), k)
    w = snn_weights(nbr)
    csr = snn_graph(nbr, w, prune)
    lab, levels = louvain(*csr, resolution)
    labels[rows] = lab
    return labels, dict(rows=rows, nbr=nbr, sim=sim, w=w, csr=csr, levels=levels)
