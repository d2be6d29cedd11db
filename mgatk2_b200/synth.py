"""Seeded synthetic 10x-ATAC-shaped chrM read batches (SURVEY.md §8d).

The reference ships no input data for this path (its test BAM is a missing blob), so every
parity test and the benchmark run on records drawn here: position-sorted paired reads with
PCR duplicates, low-mapq / secondary / supplementary / unmapped-placed records, missing and
non-whitelisted barcodes, N bases, a quality mixture and — for the stress profile — soft clips,
insertions, deletions and reads hanging over the end of chrM.

bc_idx encodes the barcode stage of readers.py:104-111 on the host side: >=0 whitelist index,
-1 no CB tag, -2 CB tag not in the whitelist (both negative values are "drop" on the device).
"""
from __future__ import annotations

import numpy as np

from .batch import ReadBatch

MITO_LENGTH = 16569

PROFILES = {
    # BASELINE.json configs[1]/[2]: 2x50 bp, CIGAR 50M
    "atac50": dict(read_len=50, softclip=0.0, ins=0.0, dele=0.0),
    # bundled-sample shape substitute (~70 bp reads)
    "atac70": dict(read_len=70, softclip=0.05, ins=0.01, dele=0.01),
    # BASELINE.json configs[4]: 2x150 bp with soft clips / indels
    "stress150": dict(read_len=150, softclip=0.20, ins=0.05, dele=0.05),
}


def make_whitelist(n_cells: int, seed: int = 0) -> list[str]:
    """`n_cells` distinct 16-mer barcodes with the 10x '-1' suffix."""
    rng = np.random.default_rng(seed ^ 0x5EED)
    out, seen = [], set()
    letters = np.array(list("ACGT"))
    while len(out) < n_cells:
        block = letters[rng.integers(0, 4, size=(n_cells - len(out) + 16, 16))]
        for row in block:
            s = "".join(row) + "-1"
            if s not in seen:
                seen.add(s)
                out.append(s)
                if len(out) == n_cells:
                    break
    return out


def _sample_categorical(rng, weights: np.ndarray, n: int) -> np.ndarray:
    cdf = np.cumsum(weights, dtype=np.float64)
    cdf /= cdf[-1]
    return np.minimum(np.searchsorted(cdf, rng.random(n), side="right"), len(weights) - 1)


_PAYLOAD_CHUNK = 1 << 17          # rows per independently seeded chunk: results do not depend on thread count


def _payload_chunk(args):
    child, rows, L = args
    rng = np.random.default_rng(child)
    Lp = L + (L & 1)
    nib_lut = np.left_shift(1, np.arange(200) & 3).astype(np.uint8)
    nib_lut[199] = 15                                     # 0.5 % N
    nib = nib_lut[rng.integers(0, 200, size=(rows, Lp), dtype=np.uint8)]
    if L & 1:
        nib[:, -1] = 0
    packed = (nib[:, 0::2] << 4) | nib[:, 1::2]
    u = np.arange(100)
    q_lut = np.where(u < 70, 40, np.where(u < 90, 25 + u % 15, 2 + u % 18)).astype(np.uint8)
    qual = q_lut[rng.integers(0, 100, size=(rows, L), dtype=np.uint8)]
    return packed, qual


def _payload(seed: int, n: int, L: int):
    """Packed 4-bit bases [n, ceil(L/2)] and qualities [n, L], drawn in row chunks on a thread pool."""
    from concurrent.futures import ThreadPoolExecutor
    import os
    n_chunks = max(1, (n + _PAYLOAD_CHUNK - 1) // _PAYLOAD_CHUNK)
    children = np.random.SeedSequence([seed, 0xB200]).spawn(n_chunks)
    jobs = [(children[k], min(_PAYLOAD_CHUNK, n - k * _PAYLOAD_CHUNK), L) for k in range(n_chunks)]
    Lp = L + (L & 1)
    packed = np.empty((n, Lp // 2), np.uint8)
    qual = np.empty((n, L), np.uint8)
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 1)) as ex:
        for k, (p, q) in enumerate(ex.map(_payload_chunk, jobs)):
            packed[k * _PAYLOAD_CHUNK: k * _PAYLOAD_CHUNK + len(p)] = p
            qual[k * _PAYLOAD_CHUNK: k * _PAYLOAD_CHUNK + len(q)] = q
    return packed, qual


def synth_batch(n_cells: int, n_records: int, profile: str = "atac50", seed: int = 20261018,
                dup_rate: float = 0.30, mito_length: int = MITO_LENGTH) -> ReadBatch:
    prof = PROFILES[profile]
    L = int(prof["read_len"])
    rng = np.random.default_rng(seed)
    P = mito_length
    n_frag = max(1, n_records // 2)

    # ---- fragments: (cell, start, insert size); 30 % copy an earlier fragment's triple ----
    cell_w = rng.lognormal(mean=0.0, sigma=1.0, size=n_cells)
    pos_bias = rng.uniform(0.25, 4.0, size=P)            # fixed seeded per-position Tn5 bias
    n_orig = max(1, int(round(n_frag * (1.0 - dup_rate))))
    cell_o = _sample_categorical(rng, cell_w, n_orig).astype(np.int32)
    start_o = _sample_categorical(rng, pos_bias, n_orig).astype(np.int64)
    isize_o = np.clip(np.rint(rng.lognormal(mean=np.log(110.0), sigma=0.55, size=n_orig)), 50, 700).astype(np.int64)
    # keep most fragments inside chrM but let ~1 % hang over the end
    over = start_o + isize_o - (P + rng.integers(0, 25, size=n_orig))
    start_o = np.where(over > 0, np.maximum(start_o - over, 0), start_o)
    src = np.concatenate([np.arange(n_orig), rng.integers(0, n_orig, size=n_frag - n_orig)])
    cell_f, start_f, isize_f = cell_o[src], start_o[src], isize_o[src]

    # per-fragment barcode fate (both mates share the tag): 2 % missing, 15 % not whitelisted
    u = rng.random(n_frag)
    bc_f = np.where(u < 0.02, -1, np.where(u < 0.17, -2, cell_f)).astype(np.int32)

    # ---- two records per fragment ----
    swap = rng.random(n_frag) < 0.5                       # which mate is read1
    fwd_flag = np.where(swap, 163, 99).astype(np.uint16)  # paired, proper, mate reverse (+read1/2)
    rev_flag = np.where(swap, 83, 147).astype(np.uint16)  # paired, proper, reverse (+read1/2)
    rev_pos = np.minimum(np.maximum(start_f + isize_f - L, 0), P - 1)
    pos = np.concatenate([start_f, rev_pos]).astype(np.int32)
    tlen = np.concatenate([isize_f, -isize_f]).astype(np.int32)
    flag = np.concatenate([fwd_flag, rev_flag])
    bc = np.concatenate([bc_f, bc_f])
    if 2 * n_frag < n_records:                            # odd request: one unpaired straggler
        pos = np.append(pos, np.int32(rng.integers(0, P)))
        tlen = np.append(tlen, np.int32(0)); flag = np.append(flag, np.uint16(0)); bc = np.append(bc, np.int32(0))
    n = len(pos)

    order = np.argsort(pos, kind="stable")
    pos, tlen, flag, bc = pos[order], tlen[order], flag[order], bc[order]

    # ---- per-record attributes, drawn in sorted order (independent of the fragment) ----
    u = rng.random(n)
    mapq = np.where(u < 0.93, 60, np.where(u < 0.96, rng.integers(30, 60, size=n), rng.integers(0, 30, size=n))).astype(np.uint8)
    u = rng.random(n)
    flag = flag | np.where(u < 0.010, 0x100, 0).astype(np.uint16)                      # secondary
    flag = flag | np.where((u >= 0.010) & (u < 0.015), 0x800, 0).astype(np.uint16)     # supplementary
    flag = flag | np.where((u >= 0.015) & (u < 0.022), 0x4, 0).astype(np.uint16)       # unmapped, placed at mate
    flag = flag | np.where((u >= 0.022) & (u < 0.030), 0x400, 0).astype(np.uint16)     # duplicate flag (ignored, Q9)

    # ---- cigars: [S] M [I|D M] [S], query-consuming lengths sum to L ----
    cat = rng.random(n)
    has_sc = cat < prof["softclip"]
    has_ins = (cat >= prof["softclip"]) & (cat < prof["softclip"] + prof["ins"])
    has_del = (cat >= prof["softclip"] + prof["ins"]) & (cat < prof["softclip"] + prof["ins"] + prof["dele"])
    sc_left = np.where(has_sc & (rng.random(n) < 0.6), rng.integers(1, min(31, L // 3), size=n), 0)
    sc_right = np.where(has_sc & ((sc_left == 0) | (rng.random(n) < 0.3)), rng.integers(1, min(31, L // 3), size=n), 0)
    indel_len = np.where(has_ins, rng.integers(1, 4, size=n), np.where(has_del, rng.integers(1, 11, size=n), 0))
    m_total = L - sc_left - sc_right - np.where(has_ins, indel_len, 0)
    m1 = np.where(has_ins | has_del, rng.integers(5, np.maximum(m_total - 5, 6)), m_total)
    m2 = m_total - m1
    words = np.zeros((n, 5), dtype=np.uint32)
    ncig = np.zeros(n, dtype=np.int64)

    def push(mask, op, length):
        rows = np.nonzero(mask)[0]
        words[rows, ncig[rows]] = (length[rows].astype(np.uint32) << 4) | np.uint32(op)
        ncig[rows] += 1

    push(sc_left > 0, 4, sc_left)
    push(np.ones(n, bool), 0, m1)
    push(has_ins, 1, indel_len)
    push(has_del, 2, indel_len)
    push(has_ins | has_del, 0, m2)
    push(sc_right > 0, 4, sc_right)

    # ---- bases (0.5 % N) and qualities {40: 70 %, 25-39: 20 %, 2-19: 10 %} ----
    Lp = L + (L & 1)
    packed, qual = _payload(seed, n, L)

    # ---- blobs: cigar | seq | qual, 16-byte aligned, laid out in record order ----
    nbytes = 4 * ncig + Lp // 2 + L
    units = (nbytes + 15) // 16
    off = np.zeros(n, dtype=np.int64)
    np.cumsum(units[:-1], out=off[1:])
    blob = np.zeros(int(units.sum()) * 16, dtype=np.uint8)
    for k in np.unique(ncig):
        rows = np.nonzero(ncig == k)[0]
        k = int(k)
        size = 4 * k + Lp // 2 + L
        mat = np.zeros((len(rows), int((size + 15) // 16) * 16), dtype=np.uint8)
        mat[:, : 4 * k] = words[rows, :k].copy().view(np.uint8).reshape(len(rows), 4 * k)
        mat[:, 4 * k: 4 * k + Lp // 2] = packed[rows]
        mat[:, 4 * k + Lp // 2: size] = qual[rows]
        if len(rows) == n:                                 # uniform batch: the matrix is the blob
            blob = mat.reshape(-1)
        else:
            b16 = blob.view("V16")
            m16 = mat.view("V16")
            for uu in range(m16.shape[1]):
                b16[off[rows] + uu] = m16[:, uu]
    return ReadBatch(pos=pos, tlen=tlen, flag=flag, mapq=mapq, bc_idx=bc,
                     l_seq=np.full(n, L, np.uint16), n_cigar=ncig.astype(np.uint16),
                     blob_off=off.astype(np.uint32), blob=blob)


def synth_deletions(n_cells: int = 40, n_fragments: int = 6000, deletions=((8470, 13446), (6330, 13994), (1500, 2100)),
                    read_len: int = 50, mito_length: int = MITO_LENGTH, seed: int = 20261022, gap_reads: bool = True,
                    n_background: int = 4000, skew: float = 0.0, het_levels=(0.0, 0.1, 0.3, 0.6, 0.9)):
    """Reads of cells that carry large deletions (1-based HGVS ranges) at chosen heteroplasmy, on a seeded reference.

    Every fragment lies at a breakpoint of one deletion. With the cell's heteroplasmy of that deletion it comes from a
    deleted molecule (ref[:l + 1] + ref[r:], l = first - 2, r = last) and crosses the junction: it is aligned on its
    longer side with a soft clip of the other side, which is added as a 0x800 supplementary record (hard-clipped). Else
    it is a wild-type read over the breakpoint; some of those end exactly at l without a clip. Per deletion there is one
    read with a D gap over the deleted segment (`gap_reads`) and two duplicates whose first copy shadows a junction read:
    one with mapq 0, one without a clip (not relevant). `n_background` plain reads cover the contig so that the reference
    vote recovers the reference; `skew` > 0 draws cells from lognormal weights of that sigma. Returns (ReadBatch, the
    reference as a string, heteroplasmy float [n_cells, D] of the draw)."""
    rng = np.random.default_rng(seed)
    P, L = int(mito_length), int(read_len)
    ref = "".join(np.array(list("ACGT"))[rng.integers(0, 4, P)])
    lr = [(int(f) - 2, int(t)) for f, t in deletions]
    D = len(lr)
    het = np.array(het_levels)[rng.integers(0, len(het_levels), size=(n_cells, max(D, 1)))][:, :D]
    w = rng.lognormal(0.0, skew, n_cells) if skew > 0 else np.ones(n_cells)
    cells = _sample_categorical(rng, w, n_fragments)
    recs = []

    def add(pos, cigar, seq, cell, flag=None, mapq=60, tlen=None):
        rev = bool(rng.random() < 0.5)
        recs.append({"pos": int(pos), "cigar": cigar, "seq": seq, "bc_idx": int(cell),
                     "flag": (147 if rev else 99) if flag is None else flag,
                     "mapq": mapq, "tlen": int((-1 if rev else 1) * rng.integers(60, 400)) if tlen is None else tlen})

    for k in range(n_fragments):
        if D == 0:
            break
        cell, d = int(cells[k]), int(rng.integers(0, D))
        l, r = lr[d]
        mq = 60 if rng.random() < 0.95 else 10
        if rng.random() < het[cell, d]:                      # deleted molecule over the junction
            a = int(rng.integers(1, L))                       # bases up to l; the other L - a from r on
            b = L - a
            seq = ref[l + 1 - a: l + 1] + ref[r: r + b]
            if a >= b:
                add(l + 1 - a, [(0, a), (4, b)], seq, cell, mapq=mq)
                add(r, [(5, a), (0, b)], ref[r: r + b], cell, flag=2048 | 0x1)
            else:
                add(r, [(4, a), (0, b)], seq, cell, mapq=mq)
                add(l + 1 - a, [(0, a), (5, b)], ref[l + 1 - a: l + 1], cell, flag=2048 | 0x1)
        else:                                                 # wild type over l / l + 1 or r - 1 / r
            at = l if rng.random() < 0.5 else r - 1
            s = at - L + 1 if (at == l and rng.random() < 0.1) else int(rng.integers(at - L + 2, at + 1))
            add(s, [(0, L)], ref[s: s + L], cell, mapq=mq)
    for d, (l, r) in enumerate(lr):
        cell = d % n_cells
        if gap_reads:
            add(l - 20, [(0, 21), (2, r - l - 1), (0, L - 21)], ref[l - 20: l + 1] + ref[r: r + L - 21], cell)
        b = L // 2
        clip_seq = ref[l + 1 - (L - b): l + 1] + ref[r: r + b]
        for first in ({"mapq": 0, "cigar": [(4, L - b), (0, b)], "seq": clip_seq},
                      {"mapq": 60, "cigar": [(0, L)], "seq": ref[r: r + L]}):
            add(r, first["cigar"], first["seq"], cell, flag=99, mapq=first["mapq"], tlen=333)
            add(r, [(4, L - b), (0, b)], clip_seq, cell, flag=99, tlen=333)        # shadowed by the one before
    for s in rng.integers(0, P - L, n_background):
        add(s, [(0, L)], ref[s: s + L], int(rng.integers(0, n_cells)), mapq=60)
    order = sorted(range(len(recs)), key=lambda i: recs[i]["pos"])          # stable: duplicates keep their order
    return ReadBatch.from_records([recs[i] for i in order]), ref, het
