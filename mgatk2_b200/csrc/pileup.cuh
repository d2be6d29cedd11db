// mgatk2_b200 — stages 4-6 of the hot path (sm_100a): per-cell, per-position, per-base, per-strand counting from the
// reference-coordinate slots (common.cuh), Tn5 sites (pileup.py:43-50), strand-bias filter / coverage / Tn5 gating
// (pileup.py:128-154) and the per-cell depth statistics, planes written once.
//
//   k_plan_scan / k_plan_units   cut every cell into position tiles ("units") of bounded read count
//   k_pileup_main                persistent CTAs, warp-specialised: a producer warp pulls units from a global counter,
//                                streams each unit's slots into shared memory with ONE bulk asynchronous copy (TMA)
//                                (full mbarrier), then builds the unit's table of candidate ranges per chunk (ready
//                                mbarrier); three units in flight per CTA; the eight consumer warps take chunks of 32
//                                positions, release a stage on its empty mbarrier and never meet at a CTA barrier
//   k_pileup_big                 the rare units that do not fit a stage (hot spots, piles beyond 65535): sub-tiles and
//                                batches, plain loads, CTA barriers
//
// Counting a chunk: the candidate reads are those starting in (chunk - extent, chunk + 32), a range of the unit's slots
// read from the table (k_pileup_main) or found by a 32-way search (k_pileup_big); 32 candidates at a time,
// one per lane: the 32-bit window of the read's three planes at offset chunk - start; a 32x32 bit transpose across the
// warp turns "lane = read" into "lane = position" for the four bit matrices of the round (V, B0, B1 and the Tn5 sites;
// one or two transposes when the candidates fit 8 or 16 lanes), and one LOP3 + popcount per base and strand adds up the
// ten counters in registers. Nothing is shared between warps, so there are no atomics on counters; when the chunk's
// reads are exhausted the counts are final.
#pragma once
#include "common.cuh"

namespace mgatk {

#ifndef MGATK_PILEUP_WARPS
#define MGATK_PILEUP_WARPS 8
#endif
constexpr int kWarpsPerCta = MGATK_PILEUP_WARPS;       // consumer warps of a pileup CTA
constexpr int kThreads = kWarpsPerCta * 32;
constexpr int kSplitChunks = 4;       // k_pileup_big "deep" units: at most this many chunks of 32 positions; their reads come in batches
constexpr int kAccWords = 10 * 32;   // deep units: counts of one chunk, [8 base x strand + 2 Tn5][32]

struct Unit { int32_t cell, t0, t1, rbeg, rend; };

// The reads to pile up (k_dedup's compacted array), cell-major, sorted by start inside a cell.
// (Listing the survivors by place instead of copying them - k_dedup writes 4 bytes per read, the pileup producer gathers
// the 32-byte slots with one bulk copy each - was measured: dedup 0.314 -> 0.268 ms, pileup 0.56 -> 1.08 ms. Rejected.)
struct SlotList {
    const uint8_t *slots; int slot_bytes;
    __device__ __forceinline__ const uint8_t *at(int64_t i) const { return slots + (size_t)i * slot_bytes; }
    __device__ __forceinline__ int pos(int64_t i) const { return *reinterpret_cast<const int32_t *>(at(i)); }
};

// ---------------------------------------------------------------------------------------------
// Work planning: a unit is (cell, position tile). Tile borders sit at every `unit_reads`-th read of
// the cell (rounded down to a chunk of 32 positions), so units carry about the same number of reads
// wherever the cell's coverage is dense or sparse. Dead cells (processors.py:22) and cells without
// reads to pile up get one unit that only writes zeros.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int tiles_for(int cnt, int unit_reads, int ppad) {
    int nt = cnt <= 0 ? 1 : (cnt + unit_reads - 1) / unit_reads;
    const int max_nt = ppad / 32;
    return nt > max_nt ? max_nt : nt;
}

__device__ __forceinline__ bool cell_dead(const mgatk_cell_qc &q, int min_reads) {
    return q.n_reads == 0 || (int64_t)q.n_reads < (int64_t)min_reads;
}

// one pass over the cells: first compacted record of every cell (exclusive scan of the per-cell counts of k_dedup)
// and first unit of every cell (exclusive scan of the tile counts), both in one 64-bit scan
__global__ void __launch_bounds__(1024)
k_plan_scan(const mgatk_cell_qc *__restrict__ qc, int n_cells, int min_reads,
            int unit_reads, int ppad, int32_t *__restrict__ cell_start, int32_t *__restrict__ unit_start, int32_t *__restrict__ n_units) {
    __shared__ u64 warp_sums[32];
    __shared__ u64 carry_s;
    const int t = threadIdx.x, lane = t & 31, wid = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n_cells; c0 += 1024) {
        const int c = c0 + t;
        u64 mine = 0;                                        // records << 32 | tiles
        if (c < n_cells) {
            const u32 np = qc[c].median_lo;                  // parked there by k_dedup
            const int cnt = cell_dead(qc[c], min_reads) ? 0 : (int)np;
            mine = ((u64)np << 32) | (u32)tiles_for(cnt, unit_reads, ppad);
        }
        u64 inc = mine;
        for (int o = 1; o < 32; o <<= 1) { const u64 v = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += v; }
        if (lane == 31) warp_sums[wid] = inc;
        __syncthreads();
        if (wid == 0) {
            const u64 v = warp_sums[lane];
            u64 sc = v;
            for (int o = 1; o < 32; o <<= 1) { const u64 x = __shfl_up_sync(kFull, sc, o); if (lane >= o) sc += x; }
            warp_sums[lane] = sc - v;
        }
        __syncthreads();
        const u64 carry = carry_s;
        const u64 excl = carry + warp_sums[wid] + inc - mine;
        if (c < n_cells) { cell_start[c] = (int32_t)(excl >> 32); unit_start[c] = (int32_t)(u32)excl; }
        __syncthreads();
        if (t == 1023) carry_s = carry + warp_sums[31] + inc;
        __syncthreads();
    }
    if (t == 0) { cell_start[n_cells] = (int32_t)(carry_s >> 32); unit_start[n_cells] = (int32_t)(u32)carry_s; *n_units = (int32_t)(u32)carry_s; }
}

#ifndef MGATK_PLAN_GALLOP
#define MGATK_PLAN_GALLOP 1
#endif
__global__ void k_plan_units(const int32_t *__restrict__ cell_start, const mgatk_cell_qc *__restrict__ qc,
                             SlotList sl, const int32_t *__restrict__ unit_start, int n_cells,
                             int min_reads, int unit_reads, int ppad, int halo, Unit *__restrict__ units,
                             int cap_reads, Unit *__restrict__ units_big, int32_t *__restrict__ n_big_units) {
    // (one warp per unit with 32 probes per search step was measured slower: 0.060 against 0.041 ms for plan on C2)
    const int u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= unit_start[n_cells]) return;
    int lo = 0, hi = n_cells;                              // last cell with unit_start[c] <= u
    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (unit_start[mid] <= u) lo = mid; else hi = mid; }
    const int c = lo;
    const bool dead = cell_dead(qc[c], min_reads);
    const int cs = cell_start[c], ce = cell_start[c + 1];
    const int cnt = dead ? 0 : ce - cs;
    const int nt = tiles_for(cnt, unit_reads, ppad), k = u - unit_start[c];
    const int per = cnt > 0 ? (cnt + nt - 1) / nt : 0;
    Unit un;
    un.cell = c;
    un.t0 = 0; un.t1 = ppad;
    if (k > 0) un.t0 = min(max(sl.pos(cs + min(k * per, cnt - 1)), 0), ppad) & ~31;
    if (k + 1 < nt) un.t1 = min(max(sl.pos(cs + min((k + 1) * per, cnt - 1)), 0), ppad) & ~31;
    if (un.t1 < un.t0) un.t1 = un.t0;
    if (cnt == 0) { un.rbeg = un.rend = 0; }
    else {
        const int first = un.t0 - halo + 1;                // reads starting before cannot reach t0
#if MGATK_PLAN_GALLOP
        // both borders sit just below the reads the tile borders were taken from (plan 0.041 -> 0.037 ms on C2)
        un.rbeg = un.t0 == 0 ? cs : lower_bound_near(sl, cs, ce, cs + min(k * per, cnt - 1), first);   // the leftmost tile also takes the reads left of 0
        un.rend = lower_bound_near(sl, cs, ce, cs + min((k + 1) * per, cnt - 1), un.t1);      // (>= rbeg: t1 >= t0 > first)
#else
        int a = cs, b = un.t0 == 0 ? cs : ce;              // the leftmost tile also takes the reads left of 0
        while (a < b) { int mid = (a + b) >> 1; if (sl.pos(mid) < first) a = mid + 1; else b = mid; }
        un.rbeg = a;
        b = ce;
        while (a < b) { int mid = (a + b) >> 1; if (sl.pos(mid) < un.t1) a = mid + 1; else b = mid; }
        un.rend = a;
#endif
    }
    // a tile with more reads than a stage of the main kernel holds (a hot spot, a deep pile) goes to the list of
    // k_pileup_big, which walks it in sub-tiles and batches
    if (un.rend - un.rbeg > cap_reads) {
        units_big[atomicAdd(n_big_units, 1)] = un;
        un.t1 = un.t0;                                      // empty here
    }
    units[u] = un;
}

struct PileupArgs {
    const uint8_t *slots;            // the reads to pile up (k_dedup), cell-major, sorted by start inside a cell
    const uint8_t *blob; int64_t blob_bytes;     // the caller's blob: indirect reads only
    const Unit *units; const int32_t *n_units; int32_t *work_counter;
    uint16_t *planes; mgatk_cell_qc *qc; mgatk_stats *stats;
    mgatk_overflow *ovf; int64_t ovf_cap;
    int P, ppad, min_baseq, dist, apply_bias, extent, raw;
    int accumulate;                  // streaming: add the counts of this batch to the planes, nothing else (MGATK_FLAG_ACCUMULATE)
    int slot_bytes, words;           // slot layout (common.cuh)
    int cap_reads;                   // slots per stage (main) / per batch (big)
    u32 *totals32;                   // [4][ppad] cross-cell base totals of this batch (fwd + rev after the filters), or null
    // streaming: cells with an entry beyond 65535 get a set of 32-bit carry planes (count of 65536-wraps per entry of the
    // ten counted planes), so accumulation stays exact for any depth; deep_map[cell] = set index, -1 none yet
    int32_t *deep_map; u32 *deep_planes; int32_t *deep_count; int deep_cap;
    double max_bias;
};

// per-lane constants of the five butterfly stages: byte selectors for j = 16, 8 (whole bytes move), keep mask and
// rotate amount for j = 4, 2, 1
struct TransposeConst { u32 sel[2], keep[3], amt[3]; };
__device__ __forceinline__ TransposeConst make_transpose_const(int lane) {
    TransposeConst tc;
    tc.sel[0] = transpose_sel(lane, 16); tc.sel[1] = transpose_sel(lane, 8);
    asm volatile("" : "+r"(tc.sel[0]), "+r"(tc.sel[1]));
#pragma unroll
    for (int s = 0; s < 3; s++) {
        tc.keep[s] = transpose_keep(lane, 4 >> s); tc.amt[s] = transpose_amt(lane, 4 >> s);
        // opaque to the compiler: it would otherwise recompute both with two SELs per stage on the saturated ALU pipe
        asm volatile("" : "+r"(tc.keep[s]), "+r"(tc.amt[s]));
    }
    return tc;
}
__device__ __forceinline__ u32 warp_transpose(u32 x, const TransposeConst &tc) {
    x = transpose_stage_bytes(x, __shfl_xor_sync(kFull, x, 16), tc.sel[0]);
    x = transpose_stage_bytes(x, __shfl_xor_sync(kFull, x, 8), tc.sel[1]);
#pragma unroll
    for (int s = 0; s < 3; s++) x = transpose_stage(x, __shfl_xor_sync(kFull, x, 4 >> s), tc.keep[s], tc.amt[s]);
    return x;
}

// The carry planes of a cell (streaming): looked up, or claimed by lane 0 when the cell has none yet. Warp-uniform call.
__device__ __forceinline__ int deep_set_of(const PileupArgs &a, int cell, int lane) {
    int set = -1;
    if (a.deep_map && lane == 0) {
        volatile int32_t *m = a.deep_map + cell;
        int s = *m;
        if (s == -1 && atomicCAS(a.deep_map + cell, -1, -2) == -1) {             // ours to claim
            const int k = atomicAdd(a.deep_count, 1);
            s = k < a.deep_cap ? k : -3;                                          // -3: every set is taken
            __threadfence();
            atomicExch(a.deep_map + cell, s);
        } else {
            while ((s = *m) == -2 || s == -1) {}                                  // another warp is claiming it
        }
        set = s >= 0 ? s : -1;
    }
    return __shfl_sync(kFull, set, 0);
}

// The counts of a chunk are final: strand-bias filter, coverage, Tn5 gating (pileup.py:128-154), depth
// statistics, saturation (writers.py:205-218) and the one write of the 11 planes. kAcc: a.accumulate, compiled in.
template <int kPpad, bool kAcc>
__device__ __forceinline__ void finish_chunk(const PileupArgs &a, int cell, int c0, int lane, u32 (&cnt)[10],
                                             u64 &sum, u32 &covered, u32 &maxd) {
    const int ppad = kPpad ? kPpad : a.ppad;             // compile-time plane pitch: the 11 stores share one address
    const int p = c0 + lane;
    if (c0 + 32 > a.P) {                             // the contig's last chunk only (warp-uniform)
#pragma unroll                                       // pileup.py:58 end_refpos = min(.., mito_length): padding stays zero
        for (int k = 0; k < 10; k++) cnt[k] = p >= a.P ? 0u : cnt[k];
    }
    if (kAcc) {                                      // streamed batches: raw counts add up in the planes; filters, coverage
        uint16_t *acc = a.planes + (size_t)cell * MGATK_N_PLANES * ppad + p;      // and statistics come in k_stream_finish
        u32 v[10], wraps = 0u;
#pragma unroll
        for (int pl = 0; pl < 10; pl++) {
            v[pl] = cnt[pl] ? (u32)acc[(size_t)pl * ppad] + cnt[pl] : 0u;
            wraps |= v[pl] >> 16;
        }
        int set = -1;
        if (__any_sync(kFull, wraps != 0u)) set = deep_set_of(a, cell, lane);      // an entry passes 65535: the cell's carry planes
        bool sat = false;
#pragma unroll
        for (int pl = 0; pl < 10; pl++) {
            if (cnt[pl]) {
                if (v[pl] > 65535u) {
                    if (set >= 0) { atomicAdd(a.deep_planes + ((size_t)set * 10 + pl) * ppad + p, v[pl] >> 16); v[pl] &= 0xffffu; }
                    else { v[pl] = 65535u; sat = true; }
                }
                acc[(size_t)pl * ppad] = (uint16_t)v[pl];
            }
        }
        if (sat) atomicOr((u64 *)&a.stats->error_bits, (u64)ERR_SATURATED);      // no carry planes (left): refused, not saturated
        return;
    }
    if (a.apply_bias) {
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const u32 f = cnt[2 * b], r = cnt[2 * b + 1], t = f + r;
            if (t > 0) {                             // pileup.py:143-148, IEEE double, strict >
                const double bias = (double)max(f, r) / (double)t;
                if (bias > a.max_bias) { cnt[2 * b] = 0; cnt[2 * b + 1] = 0; }
            }
        }
    }
    const u32 cov = ((cnt[0] + cnt[1]) + (cnt[2] + cnt[3])) + ((cnt[4] + cnt[5]) + (cnt[6] + cnt[7]));  // pileup.py:150
    if (a.totals32 && cov) {                         // reference-allele vote input (writers.py:220-222): one reduction per base,
#pragma unroll                                       // lanes = consecutive words of the base's row (exact, before saturation)
        for (int b = 0; b < 4; b++) {                // predicated RED, no branch
            const u32 t = cnt[2 * b] + cnt[2 * b + 1];
            asm volatile("{\n .reg .pred q;\n setp.ne.u32 q, %1, 0;\n @q red.global.add.u32 [%0], %1;\n}"
                         :: "l"(a.totals32 + (size_t)b * ppad + p), "r"(t) : "memory");
        }
    }
    if (cov == 0) { if (!a.raw) { cnt[8] = 0; cnt[9] = 0; } }   // pileup.py:152-153: dropped with its Tn5 counts
    else { sum += cov; covered++; maxd = max(maxd, cov); }
    u32 vals[MGATK_N_PLANES];
#pragma unroll
    for (int k = 0; k < 10; k++) vals[k] = cnt[k];
    vals[10] = cov;
    if (max(max(cov, cnt[8]), cnt[9]) > 65535u) {    // rare: exact value kept aside
#pragma unroll
        for (int pl = 0; pl < MGATK_N_PLANES; pl++) {
            if (vals[pl] > 65535u) {
                const u64 idx = atomicAdd((u64 *)&a.stats->n_overflow, 1ull);
                if ((int64_t)idx < a.ovf_cap) {
                    a.ovf[idx].cell = cell;
                    a.ovf[idx].plane_pos = ((u32)pl << 24) | (u32)p;
                    a.ovf[idx].value = vals[pl];
                } else atomicOr((u64 *)&a.stats->error_bits, (u64)ERR_OVERFLOW_CAP);
                vals[pl] = 65535u;
            }
        }
    }
    uint16_t *out = a.planes + (size_t)cell * MGATK_N_PLANES * ppad + p;
#pragma unroll
    for (int pl = 0; pl < MGATK_N_PLANES; pl++) out[(size_t)pl * ppad] = (uint16_t)vals[pl];
}
template <int kPpad>
__device__ __forceinline__ void finish_chunk_rt(const PileupArgs &a, int cell, int c0, int lane, u32 (&cnt)[10],
                                                u64 &sum, u32 &covered, u32 &maxd) {
    if (a.accumulate) finish_chunk<kPpad, true>(a, cell, c0, lane, cnt, sum, covered, maxd);
    else finish_chunk<kPpad, false>(a, cell, c0, lane, cnt, sum, covered, maxd);
}

// Per-base form of one aligned block for an indirect read (no planes in its slot): chunk bits [pa, pa + span)
// for query bases q0.. (already clipped to the distance-from-end window). m = planes V, B0, B1.
__device__ __noinline__ void block_masks_global(const uint8_t *seq, int L, int pa, int span, int q0, int min_baseq, u32 (&m)[3]) {
    const int8_t *qual = reinterpret_cast<const int8_t *>(seq) + ((L + 1) >> 1);
    const int b0 = max(pa, 0), b1 = min(pa + span, 32);
    for (int b = b0; b < b1; b++) {
        const int q = q0 + (b - pa);                           // pileup.py:75
        if ((int)__ldg(qual + q) < min_baseq) continue;        // int8 compare, pileup.py:80
        const u32 by = __ldg(seq + (q >> 1));
        const u32 nib = (q & 1) ? (by & 15u) : (by >> 4);
        const u32 bit = 1u << b;
        if (nib == 1) m[0] |= bit;                             // pileup.py:83-86: A, C, G, T only
        else if (nib == 2) { m[0] |= bit; m[1] |= bit; }
        else if (nib == 4) { m[0] |= bit; m[2] |= bit; }
        else if (nib == 8) { m[0] |= bit; m[1] |= bit; m[2] |= bit; }
    }
}

// windows of an indirect read (longer than the slot's planes) over chunk [c0, c0 + 32): CIGAR walk over the caller's blob
__device__ __noinline__ void indirect_windows(const PileupArgs &a, u32 blob_off, u32 len, int pos, int c0, u32 (&wv)[3]) {
    const int L = (int)(len & 0xffffu), ncig = (int)(len >> 16);
    const u32 *cig = reinterpret_cast<const u32 *>(a.blob + 16 * (size_t)blob_off);
    const int q_lo = a.dist > 0 ? a.dist : 0, q_hi = a.dist > 0 ? L - a.dist : L;
    const int c1 = c0 + 32;
    int ref = pos, qp = 0;
    for (int ci = 0; ci < ncig; ci++) {
        const u32 w = __ldg(cig + ci);
        const int op = w & 15;
        const int n = min((int)(w >> 4), kOpCap);
        if (cigar_op_aligned(op)) {                          // pileup.py:56
            const int va = max(q_lo - qp, 0), vb = min(min(q_hi, L) - qp, n);
            const int r0 = ref, q00 = qp;
            ref += n; qp = min(qp + n, kRefCap);              // pileup.py:90-91
            if (vb > va && r0 + va < c1 && r0 + vb > c0)
                block_masks_global(reinterpret_cast<const uint8_t *>(cig + ncig), L, r0 + va - c0, vb - va, q00 + va, a.min_baseq, wv);
        } else if (cigar_op_ref_only(op)) ref += n;          // pileup.py:92-93
        else if (op == 4) qp = min(qp + n, kRefCap);         // pileup.py:94-95; I, H, P: nothing (sic)
        if (ref >= c1) break;                                // blocks only move right
    }
}

// A slot in shared memory: start, flags, Tn5 offset and the 32-bit windows of its planes at a reference offset.
template <bool kCompact> struct SlotView;
template <> struct SlotView<true> {
    u32 w[8];
    __device__ __forceinline__ void load(u32 s) {
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(s));
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "r"(s + 16u));
    }
    __device__ __forceinline__ int pos() const { return (int)w[0]; }
    __device__ __forceinline__ u32 meta() const { return (w[3] >> 24) & 31u; }
    __device__ __forceinline__ int tn5off() const { return (int)((w[5] >> 24) & 63u); }
    __device__ __forceinline__ static u32 win(u32 lo, u32 hi24, int sh) {     // bits [sh, sh + 32) of a 56-bit plane, sh in (-32, 56]
        const u32 hi = hi24 & 0xffffffu;
        if (sh >= 32) return sh >= 56 ? 0u : hi >> (sh - 32);
        if (sh >= 0) return funnel_r(lo, hi, (u32)sh);
        return lo << (-sh);
    }
    // the same for the three planes at once and without branches (every lane of a round has its own offset, so the
    // three cases of win() would all be walked by every warp): the window is a funnel shift of two of the words
    // (0, lo, hi, 0), picked by where it starts
    __device__ __forceinline__ void window(const PileupArgs &, u32, int sh, u32 &v, u32 &b0, u32 &b1) const {
#ifdef MGATK_BRANCHY_WINDOW
        v = win(w[2], w[3], sh); b0 = win(w[4], w[5], sh); b1 = win(w[6], w[7], sh);
#else
        const u32 t = (u32)(sh + 32), s = t & 31u;           // sh in (-32, 56]: t in [1, 88]
        const bool below = t < 32u, above = t >= 64u;
#pragma unroll
        for (int k = 0; k < 3; k++) {
            const u32 lo = w[2 + 2 * k], hi = w[3 + 2 * k] & 0xffffffu;
            const u32 a = below ? 0u : (above ? hi : lo), b = below ? lo : (above ? 0u : hi);
            const u32 r = funnel_r(a, b, s);
            if (k == 0) v = r; else if (k == 1) b0 = r; else b1 = r;
        }
#endif
    }
};
template <> struct SlotView<false> {
    u32 w[4];
    __device__ __forceinline__ void load(u32 s) {
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(s));
    }
    __device__ __forceinline__ int pos() const { return (int)w[0]; }
    __device__ __forceinline__ u32 meta() const { return w[2] >> 24; }
    __device__ __forceinline__ int tn5off() const { return (int)(w[3] & 0xffffu); }
    __device__ __forceinline__ void window(const PileupArgs &a, u32 s, int sh, u32 &v, u32 &b0, u32 &b1) const {
        const SharedMem smem;
        u32 o[3] = {0u, 0u, 0u};
        if (meta() & SM_INDIRECT) {
            u32 g[4];
            smem.ld128(s + 16u, g);
            indirect_windows(a, g[0], g[1], pos(), pos() + sh, o);
        } else if (sh < 32 * a.words && sh > -32) query_window(smem, s + 16u, a.words, sh, o);
        v = o[0]; b0 = o[1]; b1 = o[2];
    }
};

// first of the n slots at `addr` (sorted by start) that starts after `key`: 32-way search across the warp
__device__ __forceinline__ int first_above(u32 addr, u32 stride, int n, int key, int lane) {
    const SharedMem smem;
    int lo = 0, hi = n;                                      // the answer lies in [lo, hi]
    while (lo < hi) {
        const int step = (hi - lo + 31) >> 5;
        const int idx = lo + lane * step;
        bool above = true;
        if (idx < hi) above = (int)smem.ld32(addr + (u32)idx * stride) > key;
        const u32 b = __ballot_sync(kFull, above);
        const int f = b ? __ffs(b) - 1 : 32;                 // first probe above the key
        if (f == 0) return lo;
        hi = min(lo + f * step, hi);
        lo = lo + (f - 1) * step + 1;
    }
    return lo;
}

// One round of a chunk's counting: the nc candidates (1 <= nc <= 32) from slot r of the slots at `addr` (shared memory),
// one per lane, are added to the counts of the 32 positions from c0 (lane = position).
template <bool kCompact>
__device__ __forceinline__ void count_round(const PileupArgs &a, u32 addr, int r, int nc, int c0, int lane,
                                            const TransposeConst &tc, u32 (&cnt)[10]) {
    u32 pv = 0u, p0 = 0u, p1 = 0u, m5 = 0u;                  // planes of this read inside the chunk: valid base, code bits, Tn5 site
    int strand = 0;
    if (lane < nc) {
        SlotView<kCompact> sv;
        const u32 s = addr + (u32)(r + lane) * (kCompact ? 32u : (u32)a.slot_bytes);
        sv.load(s);
        const int pos = sv.pos();
        strand = (sv.meta() & SM_STRAND) ? 1 : 0;
        // Tn5 site (pileup.py:43-50): reverse = start + len(SEQ) - 1, forward = start
        const int t5 = strand ? pos + sv.tn5off() : pos;
        if ((u32)(t5 - c0) < 32u && t5 < a.P) m5 = 1u << (t5 - c0);
        sv.window(a, s, c0 - pos, pv, p0, p1);
    }
    // lane = read -> lane = position. The four bit matrices of a round (V, B0, B1, Tn5; rows = reads) share one 32x32
    // transpose when there are at most 8 candidates (one matrix per byte), two when there are at most 16; forward and
    // reverse reads are counted apart (pileup.py:88)
    const u32 rev = __ballot_sync(kFull, strand);
    u32 v, b0, b1, t5;
    if (nc <= 8) {
        const int src = lane & 7;
        const u32 s0 = __shfl_sync(kFull, p0, src), s1 = __shfl_sync(kFull, p1, src), s5 = __shfl_sync(kFull, m5, src);
        quarter_columns(warp_transpose(quarter_row(lane, pv, s0, s1, s5), tc), v, b0, b1, t5);
    } else if (nc <= 16) {
        const u32 s0 = __shfl_xor_sync(kFull, p0, 16), s5 = __shfl_xor_sync(kFull, m5, 16);
        const u32 ta = warp_transpose(half_row(lane, pv, s0), tc);
        const u32 tb = warp_transpose(half_row(lane, p1, s5), tc);
        half_columns(ta, tb, v, b0, b1, t5);
    } else {
        v = warp_transpose(pv, tc); b0 = warp_transpose(p0, tc); b1 = warp_transpose(p1, tc); t5 = warp_transpose(m5, tc);
    }
    count_columns(v, b0, b1, t5, rev, cnt);
}

// Counts of the 32 positions from c0 out of the candidate slots [first, last) at `addr` (those starting in
// (c0 - extent, c0 + 32)), part `part` of `nparts` of them: lane = position on return.
template <bool kCompact>
__device__ __forceinline__ void count_range(const PileupArgs &a, u32 addr, int first, int last, int c0, int part, int nparts,
                                            int lane, const TransposeConst &tc, u32 (&cnt)[10]) {
    for (int r = first + 32 * part; r < last; r += 32 * nparts) count_round<kCompact>(a, addr, r, min(last - r, 32), c0, lane, tc, cnt);
}

// Candidate ranges of every chunk of a unit whose n slots (sorted by start) sit at `addr`, built by one warp in one pass
// over the slots: entry ch of the table at `tbl` holds the first slot starting after t0 + 32 ch - extent (low half) and
// the first slot starting at or after t0 + 32 (ch + 1) (high half). Slot i fills the entries between its predecessor's
// chunk bound and its own; the entries beyond the last slot's bounds (all of them in a unit without reads) take n,
// written by all lanes.
__device__ __forceinline__ void st_shared_u16(u32 a, int v) {
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory");
}
__device__ __forceinline__ void build_ranges(u32 addr, u32 stride, int n, int t0, int n_chunks, int extent, u32 tbl, int lane) {
    const SharedMem smem;
    int pf = -1, pb = 0;                                     // last low / high entry filled so far (high entries start at 1)
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        int kf = pf, kb = pb;                                // lanes past the last slot fill nothing
        if (i < n) {
            const int x = (int)smem.ld32(addr + (u32)i * stride) - t0;
            kf = max(min((x + extent - 1) >> 5, n_chunks - 1), -1);          // last chunk whose low entry is i (if any)
            kb = max(min(x >> 5, n_chunks), 0);
        }
        int qf = __shfl_up_sync(kFull, kf, 1), qb = __shfl_up_sync(kFull, kb, 1);
        if (lane == 0) { qf = pf; qb = pb; }
        const int last = min(n - i0, 32) - 1;
        pf = __shfl_sync(kFull, kf, last); pb = __shfl_sync(kFull, kb, last);
        for (int c = qf + 1; c <= kf; c++) st_shared_u16(tbl + 4u * c, i);
        for (int c = qb + 1; c <= kb; c++) st_shared_u16(tbl + 4u * c - 2u, i);
    }
    for (int c = pf + 1 + lane; c < n_chunks; c += 32) st_shared_u16(tbl + 4u * c, n);
    for (int c = pb + 1 + lane; c <= n_chunks; c += 32) st_shared_u16(tbl + 4u * c - 2u, n);
}

// per-cell depth statistics of a finished unit (processors.py:36-39, writers.py:187-193): hardware warp reductions
__device__ __forceinline__ void unit_statistics(const PileupArgs &a, int cell, int lane, u64 sum, u32 covered, u32 maxd) {
    if (!__any_sync(kFull, covered != 0)) return;
    u64 tot;
    if (__any_sync(kFull, (sum >> 32) != 0)) {           // cannot happen below 2^32 counted bases per lane and unit
        tot = sum;
        for (int o = 16; o; o >>= 1) tot += __shfl_xor_sync(kFull, tot, o);
    } else {
        const u32 lo = (u32)sum;
        tot = (u64)__reduce_add_sync(kFull, lo & 0xffffu) + ((u64)__reduce_add_sync(kFull, lo >> 16) << 16);
    }
    const u32 cv = __reduce_add_sync(kFull, covered), mx = __reduce_max_sync(kFull, maxd);
    if (lane == 0) {
        atomicAdd((u64 *)&a.qc[cell].sum_depth, tot);
        atomicAdd(&a.qc[cell].covered, cv);
        atomicMax(&a.qc[cell].max_depth, mx);
    }
}

#ifndef MGATK_PILEUP_CTAS
#define MGATK_PILEUP_CTAS 4            // 56 registers per thread (20 bytes of spills): measured faster than 3 CTAs of 72 registers
#endif
#ifndef MGATK_PILEUP_STAGES
#define MGATK_PILEUP_STAGES 3
#endif
#ifndef MGATK_PILEUP_HINT
#define MGATK_PILEUP_HINT 500u
#endif
#ifndef MGATK_PILEUP_WIDE_STAGES
#define MGATK_PILEUP_WIDE_STAGES 2            // wide slots: stages of 32 KB - two of them leave room for three CTAs per SM
#endif
// units in flight per CTA of the main kernel: a warp may run this far ahead of the slowest
template <bool kCompact> struct PileupStages { static constexpr int value = kCompact ? MGATK_PILEUP_STAGES : MGATK_PILEUP_WIDE_STAGES; };

// Candidate-range table of one stage of k_pileup_main: one entry per chunk of the unit. A unit spans at most ppad / 32
// chunks; the table holds chrM's 518 (2 KB per stage: four CTAs per SM still fit), and on longer contigs a unit beyond
// that searches its chunks' ranges instead.
constexpr int kMaxRangeChunks = (int)MGATK_POS_PAD(16569) / 32;
__host__ __device__ inline int range_table_chunks(int ppad) { return ppad / 32 < kMaxRangeChunks ? ppad / 32 : kMaxRangeChunks; }
__host__ __device__ inline int range_table_bytes(int ppad) { return (4 * range_table_chunks(ppad) + 15) / 16 * 16; }

// The next unit with at least one chunk from the global counter (lane 0); cell -1 when there is none left.
__device__ __forceinline__ Unit claim_unit(const PileupArgs &a, int n_units) {
    Unit un;
    for (;;) {
        const int u = atomicAdd(a.work_counter, 1);
        if (u >= n_units) { un.cell = -1; un.t0 = un.t1 = un.rbeg = un.rend = 0; return un; }
        un = a.units[u];
        if (un.t1 - un.t0 >= 32) return un;                  // else an empty tile (its reads belong to the tile before, or to k_pileup_big)
    }
}

// ---------------------------------------------------------------------------------------------
// Main kernel: every unit fits one stage. Warp kWarpsPerCta is the producer: the unit descriptor into the stage, one
// bulk copy of the unit's slots (contiguous in the compacted array) signalled on the stage's `full` barrier. Once the
// slots have landed the producer builds the stage's candidate-range table (build_ranges) and signals `ready`. Consumer
// warps wait for `ready`, take chunks as they come for them, count each from its table entry straight out of the stage,
// release the stage on `empty` (one arrival per warp) and move on to the next: no CTA-wide barrier, a slow warp only
// holds back the refill of its own stage.
// kAcc: streaming (a.accumulate), compiled in.
// ---------------------------------------------------------------------------------------------
template <bool kCompact, int kPpad, bool kAcc>
__global__ void __launch_bounds__(kThreads + 32, kCompact ? MGATK_PILEUP_CTAS : 3)     // wide slots: the walk over plane groups needs the registers
k_pileup_main(PileupArgs a, int stage_bytes) {
    constexpr int kStages = PileupStages<kCompact>::value;
    extern __shared__ __align__(128) uint8_t dyn[];          // [kStages][stage_bytes] slots, then [kStages][range_table_bytes] tables
    __shared__ __align__(8) u64 s_full[kStages], s_ready[kStages], s_empty[kStages];
    __shared__ Unit s_unit[kStages];
    __shared__ int s_next[kStages];                          // next chunk of the stage's unit to hand out
    const int lane = lane_id(), wid = threadIdx.x >> 5;
    const u32 full0 = (u32)__cvta_generic_to_shared(&s_full[0]), empty0 = (u32)__cvta_generic_to_shared(&s_empty[0]);
    const u32 ready0 = (u32)__cvta_generic_to_shared(&s_ready[0]);
    const u32 stage0 = (u32)__cvta_generic_to_shared(dyn);
    const int table_chunks = range_table_chunks(kPpad ? kPpad : a.ppad);
    constexpr bool kTableAlways = kPpad != 0 && kPpad / 32 <= kMaxRangeChunks;
    const u32 table_bytes = (u32)range_table_bytes(kPpad ? kPpad : a.ppad);
    const u32 table0 = stage0 + kStages * (u32)stage_bytes;
    const u32 stride = kCompact ? 32u : (u32)a.slot_bytes;
    if (threadIdx.x == 0) {
        for (int b = 0; b < kStages; b++) {
            mbar_init(full0 + 8u * b, 1); mbar_init(ready0 + 8u * b, 32); mbar_init(empty0 + 8u * b, kWarpsPerCta);
        }
        mbar_fence_init();
    }
    __syncthreads();
    if (wid == kWarpsPerCta) {                               // ---- producer ----
        const int n_units = *a.n_units;
        for (u32 k = 0;; k++) {
            const u32 b = k % kStages, ph = (k / kStages) & 1u;
            Unit un;
            if (lane == 0) {
                if (k >= (u32)kStages) mbar_wait_sleepy(empty0 + 8u * b, ph ^ 1u, 2000u);     // all consumer warps left the stage
                // (claiming the unit before that wait, so that its descriptor load overlaps it, was measured slower:
                // pileup 0.484 against 0.476 ms on C2)
                un = claim_unit(a, n_units);
                s_unit[b] = un;
                s_next[b] = 0;
            }
            un.cell = __shfl_sync(kFull, un.cell, 0); un.t0 = __shfl_sync(kFull, un.t0, 0); un.t1 = __shfl_sync(kFull, un.t1, 0);
            un.rbeg = __shfl_sync(kFull, un.rbeg, 0); un.rend = __shfl_sync(kFull, un.rend, 0);
            const int n = un.cell >= 0 ? un.rend - un.rbeg : 0;
            const u32 bytes = (u32)n * stride;
            const u32 dst = stage0 + b * (u32)stage_bytes, bar = full0 + 8u * b;
            if (lane == 0) {
                if (bytes) {                                 // the unit's slots are one contiguous range: one bulk copy
                    fence_proxy_async();
                    mbar_expect_tx(bar, bytes);
                    bulk_load(dst, a.slots + (size_t)un.rbeg * stride, bytes, bar);
                } else mbar_arrive(bar);
            }
            const int n_chunks = (un.t1 - un.t0) >> 5;
            if (un.cell >= 0 && n_chunks <= table_chunks) {
                mbar_wait_sleepy(bar, ph, MGATK_PILEUP_HINT);
                build_ranges(dst, stride, n, un.t0, n_chunks, a.extent, table0 + b * table_bytes, lane);
            }
            mbar_arrive(ready0 + 8u * b);                    // every lane: its own table entries are written
            if (un.cell < 0) break;
        }
        return;
    }
    // ---- consumers ----
    const TransposeConst tc = make_transpose_const(lane);
    const SharedMem smem;
    for (u32 k = 0;; k++) {
        const u32 b = k % kStages, ph = (k / kStages) & 1u;
        mbar_wait_sleepy(ready0 + 8u * b, ph, MGATK_PILEUP_HINT);
        const Unit un = s_unit[b];
        if (un.cell < 0) break;
        mbar_wait_sleepy(full0 + 8u * b, ph, MGATK_PILEUP_HINT);   // (complete already when the producer built the table)
        const u32 addr = stage0 + b * (u32)stage_bytes, tbl = table0 + b * table_bytes;
        const int n = un.rend - un.rbeg, n_chunks = (un.t1 - un.t0) >> 5;
        const bool table = kTableAlways || n_chunks <= table_chunks;
        u64 sum = 0; u32 covered = 0, maxd = 0;
        for (;;) {                                           // chunks are handed out as the warps come for them: a warp with a
            int ch = 0;                                      // crowded chunk (Tn5 hot spot) does not hold the others back
            if (lane == 0) ch = atomicAdd(&s_next[b], 1);    // (pileup 0.563 -> 0.539 ms on C2 against round-robin chunks)
            ch = __shfl_sync(kFull, ch, 0);
            if (ch >= n_chunks) break;
            const int c0 = un.t0 + 32 * ch;
            u32 cnt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // 8 base x strand counters, Tn5 fwd / rev; lane = position
            int first, last;
            if (table) {
                const u32 e = smem.ld32(tbl + 4u * ch);
                // (clamped: slots out of order, which the partition refuses, may leave entries unwritten)
                last = min((int)(e >> 16), n); first = min((int)(e & 0xffffu), last);
            } else {
                first = first_above(addr, stride, n, c0 - a.extent, lane);
                last = first_above(addr, stride, n, c0 + 31, lane);
            }
            count_range<kCompact>(a, addr, first, last, c0, 0, 1, lane, tc, cnt);
            finish_chunk<kPpad, kAcc>(a, un.cell, c0, lane, cnt, sum, covered, maxd);
        }
        unit_statistics(a, un.cell, lane, sum, covered, maxd);
        __syncwarp();
        if (lane == 0) mbar_arrive(empty0 + 8u * b);
    }
}

// Number of slots among n (sorted by start, from `base`) whose start is below `key`: every thread of the CTA counts a
// strided share, one shared-memory counter collects the warp sums.
__device__ __forceinline__ int block_count_below(const SlotList &sl, int64_t first, int n, int key, int *s_count) {
    if (threadIdx.x == 0) *s_count = 0;
    __syncthreads();
    int c = 0;
    for (int i = threadIdx.x; i < n; i += kThreads) c += sl.pos(first + i) < key;
    c = __reduce_add_sync(kFull, c);
    if (lane_id() == 0 && c) atomicAdd(s_count, c);
    __syncthreads();
    const int total = *s_count;
    __syncthreads();                                         // everybody has read it before the counter is reused
    return total;
}

// ---------------------------------------------------------------------------------------------
// The units the main kernel cannot take (more reads than a stage holds). A wide tile is walked in sub-tiles, each cut
// where the slots are full; a sub-tile that cannot be cut any narrower (a hot spot, a pile beyond 65535) is a deep unit:
// its reads come in batches, every chunk's candidates are split over `nparts` warps, partial counts meet in s_acc and
// are finished after the last batch.
// ---------------------------------------------------------------------------------------------
template <bool kCompact, int kPpad>
__global__ void __launch_bounds__(kThreads, 2)
k_pileup_big(PileupArgs a) {
    __shared__ int s_unit, s_count;
    __shared__ u32 s_acc[kSplitChunks * kAccWords];          // deep units: counts of every chunk, summed over warps and batches
    extern __shared__ __align__(128) uint8_t dyn[];          // [cap_reads] slots
    for (int e = threadIdx.x; e < kSplitChunks * kAccWords; e += blockDim.x) s_acc[e] = 0;
    const int lane = lane_id(), wid = threadIdx.x >> 5;
    const u32 addr = (u32)__cvta_generic_to_shared(dyn);
    const int n_units = *a.n_units;
    const TransposeConst tc = make_transpose_const(lane);
    const int q16 = a.slot_bytes >> 4;
    const SlotList sl{a.slots, a.slot_bytes};
    for (;;) {
        __syncthreads();                                     // previous unit fully consumed (also covers the s_acc init)
        if (threadIdx.x == 0) s_unit = atomicAdd(a.work_counter, 1);
        __syncthreads();
        const int u = s_unit;
        if (u >= n_units) break;
        const Unit un0 = a.units[u];
        if (un0.t1 - un0.t0 < 32) continue;
        const bool split = un0.rend - un0.rbeg > a.cap_reads && un0.t1 - un0.t0 > 32 * kSplitChunks;
        int sub_t0 = un0.t0, sub_r = un0.rbeg;
        for (;;) {
            Unit un = un0;
            if (split) {
                if (sub_t0 >= un0.t1) break;
                if (sub_t0 > un0.t0) {
                    __syncthreads();                         // the previous sub-tile is consumed
                    sub_r += block_count_below(sl, sub_r, un0.rend - sub_r, sub_t0 - a.extent + 1, &s_count);
                }
                un.t0 = sub_t0; un.rbeg = sub_r;
                if (un0.rend - sub_r > a.cap_reads) {
                    const int cut = min(max(sl.pos((int64_t)sub_r + a.cap_reads), 0), un0.t1) & ~31;   // first read that finds no slot
                    un.t1 = cut > sub_t0 ? cut : min(sub_t0 + 32 * kSplitChunks, un0.t1);
                    un.rend = sub_r + block_count_below(sl, sub_r, un0.rend - sub_r, un.t1, &s_count);
                }
                sub_t0 = un.t1;
            }
            const int n_chunks = (un.t1 - un.t0) >> 5;
            // more reads than slots in a tile that could still be cut: only when the input was not sorted by start (the
            // batch is refused with MGATK_ERR_UNSORTED by the partition; nothing here may run out of bounds on it)
            if (un.rend - un.rbeg > a.cap_reads && n_chunks > kSplitChunks) un.rend = un.rbeg + a.cap_reads;
            const int n_reads = un.rend - un.rbeg;
            const bool deep = n_reads > a.cap_reads;         // (then n_chunks <= kSplitChunks)
            int nparts = 1, part_shift = 0;
            if (deep) while (nparts * 2 * n_chunks <= kWarpsPerCta) { nparts *= 2; part_shift++; }
            u64 sum = 0; u32 covered = 0, maxd = 0;
            for (int rb = 0; rb == 0 || rb < n_reads; ) {
                const int nb = min(a.cap_reads, n_reads - rb);                    // reads of this batch
                __syncthreads();                             // the previous batch / sub-tile is consumed
                {
                    uint4 *s = reinterpret_cast<uint4 *>(dyn);
                    for (int e = threadIdx.x; e < nb * q16; e += kThreads) {
                        const int j = e / q16, w = e - j * q16;
                        s[e] = reinterpret_cast<const uint4 *>(sl.at((int64_t)un.rbeg + rb + j))[w];
                    }
                }
                __syncthreads();
                for (int item = wid; item < n_chunks * nparts; item += kWarpsPerCta) {
                    const int chl = item >> part_shift, part = item & (nparts - 1);
                    const int c0 = un.t0 + 32 * chl;
                    u32 cnt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
                    const int first = first_above(addr, (u32)a.slot_bytes, nb, c0 - a.extent, lane);
                    const int last = first_above(addr, (u32)a.slot_bytes, nb, c0 + 31, lane);
                    count_range<kCompact>(a, addr, first, last, c0, part, nparts, lane, tc, cnt);
                    if (deep) {
#pragma unroll
                        for (int k = 0; k < 10; k++) if (cnt[k]) atomicAdd(&s_acc[chl * kAccWords + k * 32 + lane], cnt[k]);
                    } else {
                        finish_chunk_rt<kPpad>(a, un.cell, c0, lane, cnt, sum, covered, maxd);
                    }
                }
                rb += nb > 0 ? nb : 1;
            }
            if (deep) {
                __syncthreads();                             // all partial counts are in s_acc
                if (wid < n_chunks) {
                    u32 cnt[10];
#pragma unroll
                    for (int k = 0; k < 10; k++) { cnt[k] = s_acc[wid * kAccWords + k * 32 + lane]; s_acc[wid * kAccWords + k * 32 + lane] = 0; }
                    finish_chunk_rt<kPpad>(a, un.cell, un.t0 + 32 * wid, lane, cnt, sum, covered, maxd);
                }
            }
            unit_statistics(a, un.cell, lane, sum, covered, maxd);
            if (!split) break;
        }
    }
}

}  // namespace mgatk
