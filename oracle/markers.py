"""TEST INFRASTRUCTURE — plain numpy restatement of the clone-marker ranks (DESIGN §8 "Clone markers"), not product code.

x as in oracle/clones.py; mid-ranks by a full sort of the population's x and run detection, then the exact integers
rank2[v][g] = sum of 2 * mid-rank over group g and ties[v] = sum over runs of t^3 - t, in Python ints.
"""
from __future__ import annotations

import numpy as np

from oracle.clones import allele_frequencies


def mid_ranks2(values: np.ndarray):
    """(2 * mid-rank of every value, as int64, and the sum over runs of equal values of t^3 - t)."""
    v = np.asarray(values, np.float64)
    n = len(v)
    order = np.argsort(v, kind="stable")
    s = v[order]
    starts = np.flatnonzero(np.concatenate([[True], s[1:] != s[:-1]])) if n else np.zeros(0, np.int64)
    ends = np.concatenate([starts[1:], [n]]).astype(np.int64)
    t = ends - starts
    r2 = np.empty(n, np.int64)
    r2[order] = np.repeat(2 * starts + t + 1, t)            # 2 * (s + (t + 1) / 2)
    return r2, sum(int(k) ** 3 - int(k) for k in t.tolist())


def marker_ranks(counts: np.ndarray, labels: np.ndarray, n_groups: int):
    """(rank2 uint64 [V, G], ties uint64 [V]) of uint32 counts [V, 3, C] and int labels [C]: the population is the
    cells with a label in [1, n_groups]."""
    x = allele_frequencies(counts)
    lab = np.asarray(labels, np.int64)
    inside = (lab >= 1) & (lab <= n_groups)
    V = x.shape[0]
    rank2 = np.zeros((V, n_groups), np.uint64)
    ties = np.zeros(V, np.uint64)
    for v in range(V):
        r2, tv = mid_ranks2(x[v, inside])
        ties[v] = tv
        sums = np.zeros(n_groups, np.int64)                 # at most N (N + 1) < 2^43
        np.add.at(sums, lab[inside] - 1, r2)
        rank2[v] = sums
    return rank2, ties
