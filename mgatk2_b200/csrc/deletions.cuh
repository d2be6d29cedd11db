// mgatk2_b200 — large mtDNA deletions (DESIGN §8 "Deletions"): per-cell junction / spanning read counts of given
// deletions and the soft-clip histograms breakpoints are found from, straight from a batch's SoA arrays and blobs.
//
//   k_del_prep        one CTA: checks the deletions, sorts them by l and by r (bitonic, shared memory)
//   k_del_relevance   one thread per record: stage 1, sortedness / extent checks; the CIGAR is walked only for records
//                     whose start lies within max_read_extent of a breakpoint (or all stage-1 records when discovery is
//                     on); the records that fall in a class or carry a long clip are listed, their starts marked
//   k_del_clear / k_del_insert / k_del_min   exact first-wins dedup: an open-addressing table of the listed records'
//                     keys (cell, start, strand, |tlen| or 0); every stage-1 record on a marked start takes atomicMin of
//                     its index into its key's entry, so a listed record survives iff the entry holds its own index
//   k_del_count       the survivors that pass mapq: u32 / u64 atomics (warp-aggregated) into the caller's outputs
// Only integers leave the device, so the result does not depend on the launch shape.
#pragma once
#include "common.cuh"

namespace mgatk {

constexpr int kDelThreads = 256;
constexpr int kDelK = MGATK_DEL_KMER;
constexpr int kDelMax = MGATK_DEL_MAX;
constexpr u32 ERR_DEL_RANGE = 16;                 // a deletion outside 0 <= l, l + 1 < r < P (it matches nothing)
constexpr int kDelInvalid = 0x7fffffff;           // sort key of such a deletion: beyond every read

struct __align__(16) DelEntry { u64 a, b; };     // a = cell << 32 | start; b = (|tlen| << 1 | strand) << 32 | first index

struct DelArgs {
    mgatk_batch b;
    int32_t n_cells, P, extent, min_mapq, dedup_mode, min_clip, n_del, discover;
    u32 bitmap_mask;                               // start bitmap: bit (start & mask)
    const int32_t *left, *right;                   // the caller's deletions
    int2 *by_l, *by_r;                             // scratch: {l, index} sorted by l, {r, index} sorted by r
    int32_t *dl, *dr;                              // scratch: l, r per deletion (kDelInvalid when out of range)
    u32 *n_rel, *rel, *bitmap;
    DelEntry *table; u64 table_max;
    u32 *counts; u64 *clip_hist, *clip_seq;
    u64 *error_bits;
};

struct DelGeom { int a0, a1, span, sl, sr; };

__device__ __forceinline__ GlobalBlob del_blob(const mgatk_batch &b, int64_t i) {
    const u64 off = 16ull * b.blob_off[i];
    GlobalBlob m;
    m.base = b.blob + off;
    m.avail = off < (u64)b.blob_bytes ? (u32)min((u64)b.blob_bytes - off, 0xffffffffull) : 0u;
    return m;
}

// a0, a1, span, leading / trailing soft clips (DESIGN §8 "Deletions": a clip longer than SEQ counts as 0; without an
// M/=/X op there is no clip)
__device__ __forceinline__ DelGeom del_geometry(const GlobalBlob &mem, int ncig, int pos, int L) {
    int span = 0, sl = 0, sr = 0;
    bool seen = false;
    for (int ci = 0; ci < ncig; ci++) {
        const u32 w = mem.ld32(4u * (u32)ci);
        const int op = (int)(w & 15u), n = (int)(w >> 4) < kOpCap ? (int)(w >> 4) : kOpCap;
        if (cigar_op_aligned(op)) { seen = true; sr = 0; span += n; }
        else if (cigar_op_ref_only(op)) span += n;
        else if (op == 4) { if (seen) sr += n; else sl += n; }
        if (span > kRefCap) span = kRefCap;
    }
    if (!seen || sl > L) sl = 0;
    if (!seen || sr > L) sr = 0;
    DelGeom g;
    g.a0 = pos; g.span = span; g.sl = sl; g.sr = sr;
    const long long a1 = (long long)pos + span - 1;
    g.a1 = a1 > 0x7ffffffe ? 0x7ffffffe : (int)a1;                 // below kDelInvalid
    return g;
}

// class of a read for deletion (l, r): 0 clip_left, 1 clip_right, 2 gap, 3 wt, -1 none (the classes are disjoint)
__device__ __forceinline__ int del_class(const GlobalBlob &mem, int ncig, const DelGeom &g, int l, int r, int min_clip) {
    if (g.a1 == l) return g.sr >= min_clip ? 0 : -1;
    if (g.a0 == r) return g.sl >= min_clip ? 1 : -1;
    long long ref = g.a0;
    for (int ci = 0; ci < ncig && ref <= r; ci++) {
        const u32 w = mem.ld32(4u * (u32)ci);
        const int op = (int)(w & 15u), n = (int)(w >> 4) < kOpCap ? (int)(w >> 4) : kOpCap;
        if (cigar_op_aligned(op)) {
            const long long e = ref + n;
            if ((ref <= l && l + 1 < e) || (ref <= r - 1 && r < e)) return 3;
            ref = e;
        } else if (cigar_op_ref_only(op)) {
            if (ref == l + 1 && ref + n == r) return 2;
            ref += n;
        }
    }
    return -1;
}

// first entry of a sorted {x, index} array with x >= v
__device__ __forceinline__ int del_lower(const int2 *a, int n, int v) {
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (a[mid].x < v) lo = mid + 1; else hi = mid; }
    return lo;
}

// every deletion with l or r in [a0, a1], once: f(index)
template <class F>
__device__ __forceinline__ void del_candidates(const int2 *by_l, const int2 *by_r, const int32_t *dl, int n, int a0, int a1, F &&f) {
    for (int k = del_lower(by_l, n, a0); k < n && by_l[k].x <= a1; k++) f(by_l[k].y);
    for (int k = del_lower(by_r, n, a0); k < n && by_r[k].x <= a1; k++)
        if (dl[by_r[k].y] < a0) f(by_r[k].y);
}

__device__ __forceinline__ int del_seq_base(const GlobalBlob &mem, int ncig, int q) {       // A, C, G, T -> 0..3, else -1
    const u32 a = 4u * (u32)ncig + ((u32)q >> 1);
    const u32 byte = (mem.ld32(a & ~3u) >> (8u * (a & 3u))) & 0xffu;
    const u32 nib = (q & 1) ? (byte & 15u) : (byte >> 4);
    return nib == 1 ? 0 : nib == 2 ? 1 : nib == 4 ? 2 : nib == 8 ? 3 : -1;
}

// +1 at p; lanes of the warp that add to the same address at the same time add once
template <class T>
__device__ __forceinline__ void del_add(T *p) {
    const u32 act = __activemask();
    const u32 grp = __match_any_sync(act, (u64)(uintptr_t)p);
    if (lane_id() == __ffs(grp) - 1) atomicAdd(p, (T)__popc(grp));
}

__device__ __forceinline__ bool del_stage1(const mgatk_batch &b, int64_t i, int n_cells) {
    const int bc = b.bc_idx[i];
    return (b.flag[i] & 0x904) == 0 && bc >= 0 && bc < n_cells;
}

__device__ __forceinline__ DelEntry del_key(const DelArgs &a, int64_t i) {
    const u32 cell = (u32)a.b.bc_idx[i], start = (u32)a.b.pos[i], strand = (a.b.flag[i] & 0x10) ? 1u : 0u;
    const int32_t t = a.b.tlen[i];
    const u32 tl = a.dedup_mode == MGATK_DEDUP_FRAGMENT_LENGTH ? (t < 0 ? (u32)(-(int64_t)t) : (u32)t) : 0u;
    DelEntry k;
    k.a = ((u64)cell << 32) | start;
    k.b = ((((u64)tl << 1) | strand) << 32) | 0xffffffffull;
    return k;
}

__device__ __forceinline__ u64 del_table_cap(u32 n_rel, u64 table_max) {   // power of two >= 2 n_rel, at least 1024
    u64 c = 1024;
    while (c < 2ull * n_rel) c <<= 1;
    return c < table_max ? c : table_max;
}

__device__ __forceinline__ u64 del_hash(const DelEntry &k) {
    u64 x = k.a * 0x9E3779B97F4A7C15ull ^ (k.b >> 32) * 0xC2B2AE3D27D4EB4Full;
    x ^= x >> 29; x *= 0xBF58476D1CE4E5B9ull; x ^= x >> 32;
    return x;
}

// slot of key k (inserted before): the probe ends at k or at an empty slot (-1)
__device__ __forceinline__ int64_t del_find(const DelEntry *t, u64 cap, const DelEntry &k) {
    for (u64 s = del_hash(k) & (cap - 1);; s = (s + 1) & (cap - 1)) {
        const DelEntry e = t[s];
        if (e.a == k.a && (e.b >> 32) == (k.b >> 32)) return (int64_t)s;
        if (e.a == ~0ull) return -1;
    }
}

// ---- one CTA: check and sort the deletions ----
constexpr int kDelPrepThreads = 1024;
__global__ void __launch_bounds__(kDelPrepThreads) k_del_prep(DelArgs a) {
    __shared__ u64 kl[kDelMax], kr[kDelMax];
    const int t = threadIdx.x;
    bool bad = false;
    for (int d = t; d < kDelMax; d += blockDim.x) {
        u64 vl = ~0ull, vr = ~0ull;
        if (d < a.n_del) {
            int l = a.left[d], r = a.right[d];
            if (!(l >= 0 && l + 1 < r && r < a.P)) { bad = true; l = r = kDelInvalid; }
            a.dl[d] = l; a.dr[d] = r;
            vl = ((u64)(u32)l << 32) | (u32)d;
            vr = ((u64)(u32)r << 32) | (u32)d;
        }
        kl[d] = vl; kr[d] = vr;
    }
    if (bad) atomicOr(a.error_bits, (u64)ERR_DEL_RANGE);
    __syncthreads();
    for (int k = 2; k <= kDelMax; k <<= 1)               // bitonic sort of both key arrays
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = t; i < kDelMax; i += blockDim.x) {
                const int p = i ^ j;
                if (p > i) {
                    const bool up = (i & k) == 0;
                    if ((kl[i] > kl[p]) == up) { const u64 x = kl[i]; kl[i] = kl[p]; kl[p] = x; }
                    if ((kr[i] > kr[p]) == up) { const u64 x = kr[i]; kr[i] = kr[p]; kr[p] = x; }
                }
            }
            __syncthreads();
        }
    for (int d = t; d < a.n_del; d += blockDim.x) {
        a.by_l[d] = make_int2((int)(kl[d] >> 32), (int)(kl[d] & 0xffffffffu));
        a.by_r[d] = make_int2((int)(kr[d] >> 32), (int)(kr[d] & 0xffffffffu));
    }
}

struct DelSmem { int2 by_l[kDelMax], by_r[kDelMax]; int32_t dl[kDelMax], dr[kDelMax]; };

__device__ __forceinline__ void del_load_smem(const DelArgs &a, DelSmem &sm) {
    for (int d = threadIdx.x; d < a.n_del; d += blockDim.x) {
        sm.by_l[d] = a.by_l[d]; sm.by_r[d] = a.by_r[d]; sm.dl[d] = a.dl[d]; sm.dr[d] = a.dr[d];
    }
    __syncthreads();
}

// ---- one thread per record: stage 1, checks, the list of relevant records ----
__global__ void __launch_bounds__(kDelThreads) k_del_relevance(DelArgs a) {
    __shared__ DelSmem sm;
    del_load_smem(a, sm);
    const mgatk_batch &b = a.b;
    const int lane = lane_id();
    const int64_t n = b.n_records, stride = (int64_t)gridDim.x * blockDim.x;
    bool unsorted = false, beyond = false;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {   // warp-uniform
        const int64_t i = base + lane;
        bool rel = false;
        int pos = 0;
        if (i < n) {
            pos = __ldg(&b.pos[i]);
            if (i > 0 && pos < __ldg(&b.pos[i - 1])) unsorted = true;
            if (del_stage1(b, i, a.n_cells)) {
                const int L = b.l_seq[i];
                bool walk = a.discover != 0;
                if (L > a.extent) { beyond = true; walk = false; }
                else if (!walk) {                         // a breakpoint in [pos, pos + extent - 1]
                    const long long hi = (long long)pos + a.extent - 1;
                    const int kl = del_lower(sm.by_l, a.n_del, pos), kr = del_lower(sm.by_r, a.n_del, pos);
                    walk = (kl < a.n_del && sm.by_l[kl].x <= hi) || (kr < a.n_del && sm.by_r[kr].x <= hi);
                }
                if (walk) {
                    const GlobalBlob mem = del_blob(b, i);
                    const int ncig = b.n_cigar[i];
                    const DelGeom g = del_geometry(mem, ncig, pos, L);
                    if (g.span > a.extent) beyond = true;
                    else if (g.span > 0) {
                        rel = a.discover && (g.sl >= a.min_clip || g.sr >= a.min_clip);
                        if (!rel)
                            del_candidates(sm.by_l, sm.by_r, sm.dl, a.n_del, g.a0, g.a1, [&](int d) {
                                if (!rel && del_class(mem, ncig, g, sm.dl[d], sm.dr[d], a.min_clip) >= 0) rel = true;
                            });
                    }
                }
            }
        }
        const u32 m = __ballot_sync(kFull, rel);
        if (m) {
            u32 first = 0;
            if (lane == 0) first = atomicAdd(a.n_rel, (u32)__popc(m));
            first = __shfl_sync(kFull, first, 0);
            if (rel) {
                a.rel[first + __popc(m & ((1u << lane) - 1u))] = (u32)i;
                u32 *w = a.bitmap + (((u32)pos & a.bitmap_mask) >> 5);
                const u32 bit = 1u << ((u32)pos & 31u);
                if (!(*w & bit)) atomicOr(w, bit);
            }
        }
    }
    if (unsorted) atomicOr(a.error_bits, (u64)ERR_UNSORTED);
    if (beyond) atomicOr(a.error_bits, (u64)ERR_EXTENT);
}

// ---- dedup table ----
__global__ void __launch_bounds__(kDelThreads) k_del_clear(DelArgs a) {
    const u64 cap = del_table_cap(*a.n_rel, a.table_max);
    for (u64 s = (u64)blockIdx.x * blockDim.x + threadIdx.x; s < cap; s += (u64)gridDim.x * blockDim.x) {
        DelEntry e; e.a = ~0ull; e.b = ~0ull;
        a.table[s] = e;
    }
}

__global__ void __launch_bounds__(kDelThreads) k_del_insert(DelArgs a) {
    const u32 n_rel = *a.n_rel;
    const u64 cap = del_table_cap(n_rel, a.table_max);
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < n_rel; k += gridDim.x * blockDim.x) {
        const DelEntry key = del_key(a, a.rel[k]);
        DelEntry empty; empty.a = ~0ull; empty.b = ~0ull;
        for (u64 s = del_hash(key) & (cap - 1);; s = (s + 1) & (cap - 1)) {
            const DelEntry old = atomicCAS(&a.table[s], empty, key);
            if (old.a == ~0ull || (old.a == key.a && (old.b >> 32) == (key.b >> 32))) break;
        }
    }
}

// every stage-1 record on a marked start: its index into its key's entry (the first record of a key in file order wins)
__global__ void __launch_bounds__(kDelThreads) k_del_min(DelArgs a) {
    const mgatk_batch &b = a.b;
    const u64 cap = del_table_cap(*a.n_rel, a.table_max);
    const int lane = lane_id();
    const int64_t n = b.n_records, stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31); base < n; base += stride) {
        const int64_t i = base + lane;
        int64_t slot = -1;
        if (i < n) {
            const u32 pos = (u32)__ldg(&b.pos[i]);
            if ((a.bitmap[(pos & a.bitmap_mask) >> 5] >> (pos & 31u)) & 1u)
                if (del_stage1(b, i, a.n_cells)) slot = del_find(a.table, cap, del_key(a, i));
        }
        const u32 m = __ballot_sync(kFull, slot >= 0);
        if (slot >= 0) {
            const u32 grp = __match_any_sync(m, (u64)slot);
            if (lane == __ffs(grp) - 1)                  // the group's lowest lane holds its lowest record index
                atomicMin(reinterpret_cast<u32 *>(&a.table[slot].b), (u32)i);
        }
    }
}

// ---- the survivors that pass mapq ----
__global__ void __launch_bounds__(kDelThreads) k_del_count(DelArgs a) {
    __shared__ DelSmem sm;
    del_load_smem(a, sm);
    const mgatk_batch &b = a.b;
    const u32 n_rel = *a.n_rel;
    const u64 cap = del_table_cap(n_rel, a.table_max);
    const size_t C = (size_t)a.n_cells;
    const int P = a.P;
    u64 *end_clip = a.clip_hist, *start_clip = a.clip_hist ? a.clip_hist + P : nullptr;
    u64 *end_seq = a.clip_seq, *start_seq = a.clip_seq ? a.clip_seq + (size_t)P * kDelK * 4 : nullptr;
    for (u32 k = blockIdx.x * blockDim.x + threadIdx.x; k < n_rel; k += gridDim.x * blockDim.x) {
        const u32 i = a.rel[k];
        bool keep = (int)b.mapq[i] >= a.min_mapq;
        if (keep && a.dedup_mode != MGATK_DEDUP_NONE) {
            const int64_t s = del_find(a.table, cap, del_key(a, i));
            keep = s >= 0 && (u32)(a.table[s].b & 0xffffffffu) == i;
        }
        if (!keep) continue;
        const int cell = b.bc_idx[i], L = b.l_seq[i], ncig = b.n_cigar[i];
        const GlobalBlob mem = del_blob(b, i);
        const DelGeom g = del_geometry(mem, ncig, b.pos[i], L);
        for (int pass = 0; pass < 2; pass++) {          // del_candidates, written out: the deletions with l, then r in [a0, a1]
            const int2 *by = pass ? sm.by_r : sm.by_l;
            for (int q = del_lower(by, a.n_del, g.a0); q < a.n_del && by[q].x <= g.a1; q++) {
                const int d = by[q].y;
                if (pass && sm.dl[d] >= g.a0) continue;
                const int c = del_class(mem, ncig, g, sm.dl[d], sm.dr[d], a.min_clip);
                if (c >= 0) del_add(a.counts + ((size_t)d * 4 + c) * C + cell);
            }
        }
        if (!a.discover) continue;
        if (g.sr >= a.min_clip && g.a1 >= 0 && g.a1 < P) {
            del_add(end_clip + g.a1);
            const int m = g.sr < kDelK ? g.sr : kDelK;
            for (int j = 0; j < m; j++) {
                const int base = del_seq_base(mem, ncig, L - g.sr + j);
                if (base >= 0) del_add(end_seq + ((size_t)g.a1 * kDelK + j) * 4 + base);
            }
        }
        if (g.sl >= a.min_clip && g.a0 >= 0 && g.a0 < P) {
            del_add(start_clip + g.a0);
            const int m = g.sl < kDelK ? g.sl : kDelK;
            for (int j = 0; j < m; j++) {
                const int base = del_seq_base(mem, ncig, g.sl - 1 - j);
                if (base >= 0) del_add(start_seq + ((size_t)g.a0 * kDelK + j) * 4 + base);
            }
        }
    }
}

}  // namespace mgatk
