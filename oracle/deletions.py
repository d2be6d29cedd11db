"""TEST INFRASTRUCTURE — plain-Python restatement of DESIGN §8 "Deletions" (not product code).

Record by record over `ReadBatch.record(i)`: stage 1, a dict-based first-wins dedup per barcode, the mapq gate, then
the four read classes of every deletion and the discovery histograms, written from the definitions and independently
of the kernels (csrc/deletions.cuh)."""
from __future__ import annotations

import numpy as np

K = 16                                   # MGATK_DEL_KMER
_BASE = {"A": 0, "C": 1, "G": 2, "T": 3}
_ALIGNED, _REF_ONLY = (0, 7, 8), (2, 3)


def geometry(rec: dict) -> dict:
    """a0, a1, span, sl, sr, the M/=/X blocks and the D/N gaps of a read as half-open reference intervals."""
    pos, cig, L = rec["pos"], rec["cigar"], len(rec["seq"])
    ref, blocks, gaps = pos, [], []
    for op, n in cig:
        if op in _ALIGNED:
            blocks.append((ref, ref + n))
            ref += n
        elif op in _REF_ONLY:
            gaps.append((ref, ref + n))
            ref += n
    ops = [op for op, _ in cig]
    aligned = [k for k, op in enumerate(ops) if op in _ALIGNED]
    if aligned:
        sl = sum(n for op, n in cig[: aligned[0]] if op == 4)
        sr = sum(n for op, n in cig[aligned[-1] + 1:] if op == 4)
    else:
        sl = sr = 0
    sl = 0 if sl > L else sl
    sr = 0 if sr > L else sr
    span = ref - pos
    return {"a0": pos, "a1": pos + span - 1, "span": span, "sl": sl, "sr": sr, "blocks": blocks, "gaps": gaps}


def read_class(g: dict, l: int, r: int, min_clip: int = 5):
    """'clip_left', 'clip_right', 'gap', 'wt' or None."""
    found = []
    if g["a1"] == l and g["sr"] >= min_clip:
        found.append("clip_left")
    if g["a0"] == r and g["sl"] >= min_clip:
        found.append("clip_right")
    if (l + 1, r) in g["gaps"]:
        found.append("gap")
    if any((s <= l and l + 1 < e) or (s <= r - 1 and r < e) for s, e in g["blocks"]):
        found.append("wt")
    assert len(found) <= 1, found                 # the classes are disjoint
    return found[0] if found else None


def survivors(batch, n_cells: int, dedup_mode: int, min_mapq: int) -> list:
    """Indices of the reads the pileup counts: stage 1, first-wins dedup per barcode, then mapq (Q2)."""
    seen, out = set(), []
    for i in range(batch.n_records):
        flag, cell = int(batch.flag[i]), int(batch.bc_idx[i])
        if flag & 0x904 or not 0 <= cell < n_cells:
            continue
        if dedup_mode != 2:
            t = int(batch.tlen[i])
            key = (cell, int(batch.pos[i]), bool(flag & 0x10), abs(t) if dedup_mode == 0 else 0)
            if key in seen:
                continue
            seen.add(key)
        if int(batch.mapq[i]) >= min_mapq:
            out.append(i)
    return out


def scan(parts, n_cells: int, mito_length: int, deletions, dedup_mode: int = 0, min_mapq: int = 30,
         min_clip: int = 5, find: bool = False) -> dict:
    """counts uint32 [D, 4, C] (clip_left, clip_right, gap, wt) and, with `find`, end_clip / start_clip uint64 [P] and
    end_seq / start_seq uint64 [P, K, 4] over the parts (each one dedups on its own: they are cut on start borders)."""
    P = mito_length
    dels = [(int(l), int(r)) for l, r in deletions]
    counts = np.zeros((len(dels), 4, n_cells), np.uint32)
    hist = {k: np.zeros(P, np.uint64) for k in ("end_clip", "start_clip")}
    seq = {k: np.zeros((P, K, 4), np.uint64) for k in ("end_seq", "start_seq")}
    classes = ("clip_left", "clip_right", "gap", "wt")
    for batch in ([parts] if hasattr(parts, "n_records") else parts):
        for i in survivors(batch, n_cells, dedup_mode, min_mapq):
            rec = batch.record(i)
            g = geometry(rec)
            if g["span"] == 0:
                continue
            cell, s, L = rec["bc_idx"], rec["seq"], len(rec["seq"])
            for d, (l, r) in enumerate(dels):
                c = read_class(g, l, r, min_clip)
                if c is not None:
                    counts[d, classes.index(c), cell] += 1
            if not find:
                continue
            if g["sr"] >= min_clip and 0 <= g["a1"] < P:
                hist["end_clip"][g["a1"]] += 1
                for j in range(min(K, g["sr"])):
                    b = _BASE.get(s[L - g["sr"] + j])
                    if b is not None:
                        seq["end_seq"][g["a1"], j, b] += 1
            if g["sl"] >= min_clip and 0 <= g["a0"] < P:
                hist["start_clip"][g["a0"]] += 1
                for j in range(min(K, g["sl"])):
                    b = _BASE.get(s[g["sl"] - 1 - j])
                    if b is not None:
                        seq["start_seq"][g["a0"], j, b] += 1
    out = {"counts": counts}
    if find:
        out.update(hist)
        out.update(seq)
    return out
