// mgatk2_b200 — variant statistics (include/mgatk2_b200.h, mgatk_variant_sums; DESIGN §8 "Variant statistics").
//
// A reduction over cells for every position of the filtered planes of a result: per variant p ref>b (b != ref[p],
// ref[p] != N) the exact integer sums of mgatk_variant_sums, then dev_sum / dev_sq around the exact mean.
//
//   * one CTA owns kVarTile = 32 positions (one per lane) for every selected cell; its kVarWarps warps stride over the
//     cells, so every load of a plane row is a coalesced 64-byte read of 32 positions of one cell;
//   * pass 1 accumulates the integer fields in registers, the warps' partials are added in shared memory in warp
//     order; the CTA then knows each variant's mean exactly, and pass 2 over the same cells accumulates dev_sum /
//     dev_sq, again added in warp order. No atomics and no cross-CTA reduction: the integer fields do not depend on
//     the launch configuration and the float fields are the same bits on every run;
//   * a load that reads 65535 looks the exact value up in a hash table of the overflow list (built once per call in
//     handle scratch by k_ovf_clear / k_ovf_insert, sized from the device-side n_overflow; an empty list skips it).
#pragma once
#include "common.cuh"

namespace mgatk {

constexpr int kVarWarps = 8;
constexpr int kVarTile = 32;

// ---------------------------------------------------------------------------------------------
// overflow lookup: open addressing over key (cell + 1) << 32 | plane << 24 | pos, key 0 = empty slot
// ---------------------------------------------------------------------------------------------
struct OvfSlot { u64 key; u32 value; u32 pad; };

// slots of the table for n entries: the smallest power of two >= 2 n, at least 64 (n = 0: no table)
__host__ __device__ inline u64 ovf_table_slots(u64 n) {
    u64 s = 64;
    while (s < 2 * n) s <<= 1;
    return s;
}

__device__ __forceinline__ u64 ovf_entries(const mgatk_stats *stats, int64_t cap) {
    const u64 n = stats->n_overflow;
    return n < (u64)cap ? n : (u64)cap;
}

__device__ __forceinline__ u32 ovf_hash(u64 key, u64 mask) { return (u32)(((key * 0x9E3779B97F4A7C15ull) >> 29) & mask); }

__global__ void k_ovf_clear(OvfSlot *table, const mgatk_stats *stats, int64_t cap) {
    const u64 n = ovf_entries(stats, cap);
    if (n == 0) return;
    const u64 slots = ovf_table_slots(n);
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < slots; i += (u64)gridDim.x * blockDim.x) table[i].key = 0;
}

__global__ void k_ovf_insert(OvfSlot *table, const mgatk_overflow *ovf, const mgatk_stats *stats, int64_t cap) {
    const u64 n = ovf_entries(stats, cap);
    const u64 mask = ovf_table_slots(n) - 1;
    for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
        const mgatk_overflow o = ovf[i];
        const u64 key = ((u64)(u32)(o.cell + 1) << 32) | o.plane_pos;
        for (u32 j = ovf_hash(key, mask);; j = (j + 1) & (u32)mask) {
            const u64 prev = atomicCAS(&table[j].key, 0ull, key);
            if (prev == 0 || prev == key) { table[j].value = o.value; break; }
        }
    }
}

struct OvfTable {
    const OvfSlot *t;    // nullptr: no saturated entry has a list entry
    u32 mask;
    __device__ __forceinline__ void init(const OvfSlot *table, const mgatk_stats *stats, int64_t cap) {
        const u64 n = table ? ovf_entries(stats, cap) : 0;
        t = n ? table : nullptr;
        mask = (u32)(ovf_table_slots(n) - 1);
    }
    __device__ __forceinline__ u32 fix(u32 v, int cell, int plane, int pos) const {
        if (v != 65535u || !t) return v;
        const u64 key = ((u64)(u32)(cell + 1) << 32) | ((u32)plane << 24) | (u32)pos;
        for (u32 j = ovf_hash(key, mask);; j = (j + 1) & mask) {
            const u64 k = t[j].key;
            if (k == key) return t[j].value;
            if (k == 0) return v;                            // saturated entry without a list entry: really 65535
        }
    }
};

// ---------------------------------------------------------------------------------------------
// variant sums
// ---------------------------------------------------------------------------------------------
struct VarArgs {
    const uint16_t *planes;
    const mgatk_stats *stats;
    const int64_t *totals;
    const OvfSlot *table;
    int64_t ovf_cap;
    const uint8_t *mask;
    int C, P, ppad;
    u32 low;                       // L, >= 1
    mgatk_variant_sums *out;
};

struct AltAcc {                    // one variant's integer sums over some cells
    u64 sf, sr, ff, rr, fr, mx_a, mx_d;
    u32 det, conf, over[4];
    int mx_cell;                   // -1: no cell with d > 0 yet
};

// first of A,C,G,T with the largest total, -1 (N) when none is positive (PileupResult.reference_alleles)
__device__ __forceinline__ int ref_allele(const int64_t *totals, int p) {
    int best = 0;
    int64_t bv = totals[(size_t)p * 4];
    for (int b = 1; b < 4; b++) {
        const int64_t v = totals[(size_t)p * 4 + b];
        if (v > bv) { bv = v; best = b; }
    }
    return bv > 0 ? best : -1;
}

// a1 / d1 > a2 / d2 for d1, d2 > 0, exactly (128-bit cross products)
__device__ __forceinline__ bool frac_greater(u64 a1, u64 d1, u64 a2, u64 d2) {
    const u64 xh = __umul64hi(a1, d2), xl = a1 * d2, yh = __umul64hi(a2, d1), yl = a2 * d1;
    return xh != yh ? xh > yh : xl > yl;
}
__device__ __forceinline__ bool frac_equal(u64 a1, u64 d1, u64 a2, u64 d2) {
    return __umul64hi(a1, d2) == __umul64hi(a2, d1) && a1 * d2 == a2 * d1;
}

// candidate (a, d, cell) replaces the current maximum: larger a / d, on a tie the lower cell
__device__ __forceinline__ void max_merge(AltAcc &x, u64 a, u64 d, int cell) {
    if (cell < 0) return;
    if (x.mx_cell < 0 || frac_greater(a, d, x.mx_a, x.mx_d) || (frac_equal(a, d, x.mx_a, x.mx_d) && cell < x.mx_cell)) {
        x.mx_a = a; x.mx_d = d; x.mx_cell = cell;
    }
}

struct VarTileSmem {
    AltAcc alt[kVarTile][3];
    u64 sum_cov[kVarTile];
    u32 n_cov[kVarTile], n_low[kVarTile];
    double dev_sum[kVarTile][3], dev_sq[kVarTile][3];
};

__global__ void __launch_bounds__(kVarWarps * 32) k_variant_stats(VarArgs a) {
    __shared__ VarTileSmem sm;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = blockIdx.x * kVarTile + lane;            // < ppad: the pitch is a multiple of 64
    OvfTable ov;
    ov.init(a.table, a.stats, a.ovf_cap);
    const int ref = p < a.P ? ref_allele(a.totals, p) : -1;
    int alt[3];
#pragma unroll
    for (int j = 0; j < 3; j++) alt[j] = j + (ref >= 0 && j >= ref ? 1 : 0);
    const size_t cell_pitch = (size_t)MGATK_N_PLANES * a.ppad;

    // ---- pass 1: integer sums ----
    AltAcc acc[3];
#pragma unroll
    for (int j = 0; j < 3; j++) {
        acc[j].sf = acc[j].sr = acc[j].ff = acc[j].rr = acc[j].fr = acc[j].mx_a = acc[j].mx_d = 0;
        acc[j].det = acc[j].conf = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) acc[j].over[k] = 0;
        acc[j].mx_cell = -1;
    }
    u64 sum_cov = 0;
    u32 n_cov = 0, n_low = 0;
    for (int c = warp; c < a.C; c += kVarWarps) {
        if (a.mask && !a.mask[c]) continue;
        const uint16_t *row = a.planes + (size_t)c * cell_pitch + p;
        const u32 d = ov.fix(__ldg(row + (size_t)MGATK_PLANE_COVERAGE * a.ppad), c, MGATK_PLANE_COVERAGE, p);
        u32 f[3], r[3];
#pragma unroll
        for (int j = 0; j < 3; j++) {
            f[j] = ov.fix(__ldg(row + (size_t)(2 * alt[j]) * a.ppad), c, 2 * alt[j], p);
            r[j] = ov.fix(__ldg(row + (size_t)(2 * alt[j] + 1) * a.ppad), c, 2 * alt[j] + 1, p);
        }
        sum_cov += d;
        n_cov += d > 0;
        n_low += d < a.low;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const u64 fj = f[j], rj = r[j], aj = fj + rj;
            AltAcc &x = acc[j];
            x.sf += fj; x.sr += rj;
            x.ff += fj * fj; x.rr += rj * rj; x.fr += fj * rj;     // zero for cells with a = 0
            x.det += aj > 0;
            x.conf += (fj >= 2) & (rj >= 2);
            if (d > 0) {
                const u64 h = 100 * aj;
                x.over[0] += h >= 5ull * d; x.over[1] += h >= 10ull * d; x.over[2] += h >= 20ull * d; x.over[3] += h >= 95ull * d;
                max_merge(x, aj, d, c);                           // cells ascend within a thread: ties keep the first
            }
        }
    }
    for (int w = 0; w < kVarWarps; w++) {                   // warp partials, added in warp order
        if (warp == w) {
            if (w == 0) { sm.sum_cov[lane] = sum_cov; sm.n_cov[lane] = n_cov; sm.n_low[lane] = n_low; }
            else { sm.sum_cov[lane] += sum_cov; sm.n_cov[lane] += n_cov; sm.n_low[lane] += n_low; }
#pragma unroll
            for (int j = 0; j < 3; j++) {
                AltAcc &s = sm.alt[lane][j];
                const AltAcc &x = acc[j];
                if (w == 0) { s = x; continue; }
                s.sf += x.sf; s.sr += x.sr; s.ff += x.ff; s.rr += x.rr; s.fr += x.fr;
                s.det += x.det; s.conf += x.conf;
#pragma unroll
                for (int k = 0; k < 4; k++) s.over[k] += x.over[k];
                AltAcc m = s;
                max_merge(m, x.mx_a, x.mx_d, x.mx_cell);
                s.mx_a = m.mx_a; s.mx_d = m.mx_d; s.mx_cell = m.mx_cell;
            }
        }
        __syncthreads();
    }

    // ---- pass 2: deviations from the exact mean ----
    double mean[3], ds[3] = {0, 0, 0}, dq[3] = {0, 0, 0};
    {
        const u64 cov = sm.sum_cov[lane];
#pragma unroll
        for (int j = 0; j < 3; j++)
            mean[j] = cov ? __ddiv_rn((double)(sm.alt[lane][j].sf + sm.alt[lane][j].sr), (double)cov) : 0.0;
    }
    for (int c = warp; c < a.C; c += kVarWarps) {
        if (a.mask && !a.mask[c]) continue;
        const uint16_t *row = a.planes + (size_t)c * cell_pitch + p;
        const u32 d = ov.fix(__ldg(row + (size_t)MGATK_PLANE_COVERAGE * a.ppad), c, MGATK_PLANE_COVERAGE, p);
        if (d < a.low) continue;                            // u = 0
        const double dd = (double)d;
#pragma unroll
        for (int j = 0; j < 3; j++) {
            const u32 f = ov.fix(__ldg(row + (size_t)(2 * alt[j]) * a.ppad), c, 2 * alt[j], p);
            const u32 r = ov.fix(__ldg(row + (size_t)(2 * alt[j] + 1) * a.ppad), c, 2 * alt[j] + 1, p);
            const double u = __dsub_rn(__ddiv_rn((double)((u64)f + r), dd), mean[j]);
            ds[j] = __dadd_rn(ds[j], u);
            dq[j] = __dadd_rn(dq[j], __dmul_rn(u, u));
        }
    }
    for (int w = 0; w < kVarWarps; w++) {
        if (warp == w) {
#pragma unroll
            for (int j = 0; j < 3; j++) {
                sm.dev_sum[lane][j] = w == 0 ? ds[j] : __dadd_rn(sm.dev_sum[lane][j], ds[j]);
                sm.dev_sq[lane][j] = w == 0 ? dq[j] : __dadd_rn(sm.dev_sq[lane][j], dq[j]);
            }
        }
        __syncthreads();
    }

    // ---- out[p][alt] ----
    for (int t = threadIdx.x; t < kVarTile * 4; t += blockDim.x) {
        const int lp = t >> 2, b = t & 3, q = blockIdx.x * kVarTile + lp;
        if (q >= a.P) continue;
        const int rq = ref_allele(a.totals, q);
        mgatk_variant_sums o;
        memset(&o, 0, sizeof(o));
        o.ref = rq;
        if (rq >= 0 && b != rq) {
            const int j = b - (b > rq ? 1 : 0);
            const AltAcc &s = sm.alt[lp][j];
            o.sum_fwd = s.sf; o.sum_rev = s.sr; o.sum_cov = sm.sum_cov[lp];
            o.sum_ff = s.ff; o.sum_rr = s.rr; o.sum_fr = s.fr;
            o.max_alt = s.mx_a; o.max_cov = s.mx_d;
            o.dev_sum = sm.dev_sum[lp][j]; o.dev_sq = sm.dev_sq[lp][j];
            o.n_covered = sm.n_cov[lp]; o.n_detected = s.det; o.n_conf_detected = s.conf; o.n_strand = s.det;
            for (int k = 0; k < 4; k++) o.n_over[k] = s.over[k];
            o.n_low = sm.n_low[lp];
            o.valid = 1;
        }
        a.out[(size_t)q * 4 + b] = o;
    }
}

// ---------------------------------------------------------------------------------------------
// per-cell counts of a list of variants: out[v][0..2][c] = alt forward, alt reverse, coverage
// ---------------------------------------------------------------------------------------------
__global__ void k_variant_cells(const uint16_t *planes, const OvfSlot *table, const mgatk_stats *stats, int64_t ovf_cap,
                                const int32_t *variants, int n_variants, int C, int P, int ppad, u32 *out) {
    OvfTable ov;
    ov.init(table, stats, ovf_cap);
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const uint16_t *row = planes + (size_t)c * MGATK_N_PLANES * ppad;
    for (int v = blockIdx.y; v < n_variants; v += gridDim.y) {
        const int id = variants[v];
        u32 f = 0, r = 0, d = 0;
        if (id >= 0 && id < 4 * P) {
            const int pos = id >> 2, b = id & 3;
            f = ov.fix(__ldg(row + (size_t)(2 * b) * ppad + pos), c, 2 * b, pos);
            r = ov.fix(__ldg(row + (size_t)(2 * b + 1) * ppad + pos), c, 2 * b + 1, pos);
            d = ov.fix(__ldg(row + (size_t)MGATK_PLANE_COVERAGE * ppad + pos), c, MGATK_PLANE_COVERAGE, pos);
        }
        u32 *o = out + (size_t)v * 3 * C + c;
        o[0] = f; o[(size_t)C] = r; o[2 * (size_t)C] = d;
    }
}

}  // namespace mgatk
