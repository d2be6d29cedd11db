// mgatk2_b200 — passes over finished planes: reference-allele totals (writers.py:220-222), median depth
// (writers.py:190), the stand-alone strand-bias filter (pileup.py:128-154) and the finish pass of the streaming mode.
#pragma once
#include "pileup.cuh"

namespace mgatk {

// ---------------------------------------------------------------------------------------------
// Reference-allele vote input (writers.py:220-222): per position and base, the sum over cells of
// fwd+rev after filtering. One thread owns two positions and a group of 32 cells.
// ---------------------------------------------------------------------------------------------
constexpr int kTotalsCellGroup = 32;
__global__ void __launch_bounds__(128)
k_base_totals(const uint16_t *__restrict__ planes, int n_cells, int P, int ppad, u64 *__restrict__ totals) {
    const int pp = blockIdx.x * blockDim.x + threadIdx.x;          // position pair
    if (2 * pp >= ppad) return;
    for (int c0 = blockIdx.y * kTotalsCellGroup; c0 < n_cells; c0 += gridDim.y * kTotalsCellGroup) {   // (grid.y is capped at 65535)
    const int c1 = min(n_cells, c0 + kTotalsCellGroup);
    u32 s[4][2] = {};
    for (int c = c0; c < c1; c++) {
        const u32 *row = reinterpret_cast<const u32 *>(planes + (size_t)c * MGATK_N_PLANES * ppad) + pp;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const u32 f = __ldg(row + (size_t)(2 * b) * (ppad / 2)), r = __ldg(row + (size_t)(2 * b + 1) * (ppad / 2));
            s[b][0] += (f & 0xffff) + (r & 0xffff);
            s[b][1] += (f >> 16) + (r >> 16);
        }
    }
#pragma unroll
    for (int k = 0; k < 2; k++) {
        const int p = 2 * pp + k;
        if (p < P)
#pragma unroll
            for (int b = 0; b < 4; b++) if (s[b][k]) atomicAdd(&totals[(size_t)p * 4 + b], (u64)s[b][k]);
    }
    }
}

// the totals k_pileup reduced while counting ([4][ppad] u32: a batch holds fewer than 2^31 records) -> int64 [P][4]
__global__ void k_totals_widen(const u32 *__restrict__ t32, int P, int ppad, u64 *__restrict__ totals) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    ulonglong2 lo, hi;
    lo.x = t32[p]; lo.y = t32[(size_t)ppad + p]; hi.x = t32[(size_t)2 * ppad + p]; hi.y = t32[(size_t)3 * ppad + p];
    reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p] = lo;
    reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p + 1] = hi;
}

__global__ void k_base_totals_overflow(const mgatk_overflow *__restrict__ ovf, const mgatk_stats *__restrict__ stats,
                                       int64_t cap, int P, u64 *__restrict__ totals) {
    const int64_t n = min((int64_t)stats->n_overflow, cap);
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const int pl = ovf[k].plane_pos >> 24, p = ovf[k].plane_pos & 0xffffff;
        if (pl < 8 && p < P) atomicAdd(&totals[(size_t)p * 4 + pl / 2], (u64)(ovf[k].value - 65535u));
    }
}

// ---------------------------------------------------------------------------------------------
// PileupGenerator.filter_strand_bias (pileup.py:128-154) as a stand-alone pass over raw planes.
// ---------------------------------------------------------------------------------------------
template <class T>                                           // T = uint16_t (saturating coverage) or uint32_t (exact)
__global__ void __launch_bounds__(256)
k_filter_planes(T *__restrict__ planes, int n_cells, int P, int ppad, double max_bias) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    for (int c = blockIdx.y; c < n_cells; c += gridDim.y) {  // (grid.y is capped at 65535 blocks)
        T *row = planes + (size_t)c * MGATK_N_PLANES * ppad + p;
        u32 cov = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            u32 f = row[(size_t)(2 * b) * ppad], r = row[(size_t)(2 * b + 1) * ppad];
            const u32 t = f + r;
            if (t > 0) {
                const double bias = (double)max(f, r) / (double)t;
                if (bias > max_bias) { f = 0; r = 0; row[(size_t)(2 * b) * ppad] = 0; row[(size_t)(2 * b + 1) * ppad] = 0; }
            }
            cov += f + r;
        }
        row[(size_t)MGATK_PLANE_COVERAGE * ppad] = sizeof(T) == 2 ? (T)min(cov, 65535u) : (T)cov;
        if (cov == 0) { row[(size_t)MGATK_PLANE_TN5_FWD * ppad] = 0; row[(size_t)MGATK_PLANE_TN5_REV * ppad] = 0; }
    }
}

// ---------------------------------------------------------------------------------------------
// Streaming (batches cut on reference_start borders, planes resident and accumulating): the per-batch kernels only add
// raw counts; this pass turns the accumulated planes into the final ones exactly as a one-batch run would have written
// them: cell gate (processors.py:22), strand-bias filter, coverage, Tn5 gating (pileup.py:128-154), depth statistics.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_stream_finish(PileupArgs a, int n_cells, int min_reads) {
    const int lane = lane_id();
    const int warps = (int)((gridDim.x * (size_t)blockDim.x) >> 5), gw = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int chunks = a.ppad >> 5;
    for (long long w = gw; w < (long long)n_cells * chunks; w += warps) {
        const int cell = (int)(w / chunks), ch = (int)(w - (long long)cell * chunks);
        const bool dead = cell_dead(a.qc[cell], min_reads);
        const uint16_t *in = a.planes + (size_t)cell * MGATK_N_PLANES * a.ppad + 32 * ch + lane;
        u32 cnt[10];
        const int set = a.deep_map ? a.deep_map[cell] : -1;                       // carry planes of a deep cell: 65536-wraps per entry
#pragma unroll
        for (int k = 0; k < 10; k++) {
            cnt[k] = dead ? 0u : (u32)in[(size_t)k * a.ppad];
            if (set >= 0 && !dead) cnt[k] += a.deep_planes[((size_t)set * 10 + k) * a.ppad + 32 * ch + lane] << 16;
        }
        u64 sum = 0; u32 covered = 0, maxd = 0;
        finish_chunk<0, false>(a, cell, 32 * ch, lane, cnt, sum, covered, maxd);
        if (__any_sync(kFull, covered != 0)) {
            u64 tot = sum;
            for (int o = 16; o; o >>= 1) tot += __shfl_xor_sync(kFull, tot, o);
            const u32 cv = __reduce_add_sync(kFull, covered), mx = __reduce_max_sync(kFull, maxd);
            if (lane == 0) {
                atomicAdd((u64 *)&a.qc[cell].sum_depth, tot);
                atomicAdd(&a.qc[cell].covered, cv);
                atomicMax(&a.qc[cell].max_depth, mx);
            }
        }
    }
}

// k_dedup parks the per-cell count of reads to pile up in median_lo: cleared before every streamed batch
__global__ void k_clear_parked(mgatk_cell_qc *__restrict__ qc, int n_cells) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < n_cells) qc[c].median_lo = 0;
}

// ---------------------------------------------------------------------------------------------
// Median depth over covered positions (writers.py:190): the two middle order statistics by a
// two-level (high byte, low byte) counting select on the coverage plane. One CTA per cell.
// The plane is saturated at 65535; a cell whose deepest position lies above that (bulk mode, a deep
// pile) has the exact depths of its saturated positions in the overflow list: an order statistic that
// falls among them is selected there (radix select over the 32-bit values, one byte per pass), so the
// medians are exact whatever the depth (np.median of the unsaturated depths in the reference).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 median_scan(const u32 *hist, u32 rem, u32 &bin) {      // first bin with cumulative count > rem; returns rem inside it
    u32 acc = 0;
    for (int b = 0; b < 256; b++) { if (rem < acc + hist[b]) { bin = b; return rem - acc; } acc += hist[b]; }
    bin = 255;
    return 0;
}

// The same by one warp (every lane calls it, every lane gets the result): eight bins per lane, a warp scan of the lane
// sums, and the lane that holds the answer walks its eight bins. `total` = sum of all 256 bins.
__device__ __forceinline__ u32 median_scan_warp(const u32 *hist, u32 rem, u32 &bin, u32 &total, int lane) {
    const uint4 a = reinterpret_cast<const uint4 *>(hist)[2 * lane], b = reinterpret_cast<const uint4 *>(hist)[2 * lane + 1];
    const u32 c[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    u32 sum = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) sum += c[q];
    u32 inc = sum;
    for (int o = 1; o < 32; o <<= 1) { const u32 v = __shfl_up_sync(kFull, inc, o); if (lane >= o) inc += v; }
    total = __shfl_sync(kFull, inc, 31);
    const u32 holds = __ballot_sync(kFull, inc > rem);     // lanes whose bins reach beyond rank `rem`
    if (!holds) { bin = 255; return 0; }
    const int L = __ffs(holds) - 1;
    u32 acc = inc - sum, fb = 0, fr = 0;
    bool found = false;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        if (!found && rem < acc + c[q]) { fb = 8u * (u32)lane + (u32)q; fr = rem - acc; found = true; }
        acc += c[q];
    }
    bin = __shfl_sync(kFull, fb, L);
    return __shfl_sync(kFull, fr, L);
}

#ifndef MGATK_MEDIAN_V2
#define MGATK_MEDIAN_V2 1
#endif
#if MGATK_MEDIAN_V2
// Depths below 256 - nearly all of them - get an exact histogram in the first pass (`fine`), deeper ones are counted by
// their high byte (`hist`): a median below 256 is read off `fine` at once, only a deeper one needs the second pass over
// the plane (low bytes inside its high-byte bin). The selections are made by one warp (median_scan_warp).
__global__ void __launch_bounds__(256)
k_median(const uint16_t *__restrict__ planes, int P, int ppad, mgatk_cell_qc *__restrict__ qc,
         const mgatk_overflow *__restrict__ ovf, const mgatk_stats *__restrict__ stats, int64_t ovf_cap,
         const u32 *__restrict__ t32, u64 *__restrict__ totals) {
    if (t32)                                                 // the base totals the pileup kernel reduced, widened to int64 [P][4] (k_totals_widen)
        for (int p = blockIdx.x * 256 + threadIdx.x; p < P; p += gridDim.x * 256) {
            ulonglong2 lo, hi;
            lo.x = t32[p]; lo.y = t32[(size_t)ppad + p]; hi.x = t32[(size_t)2 * ppad + p]; hi.y = t32[(size_t)3 * ppad + p];
            reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p] = lo;
            reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p + 1] = hi;
        }
    __shared__ __align__(16) u32 hist[256];                  // depths >= 256 by high byte; later: scratch of the second pass / the list
    // depths 1..255, four copies picked by lane (neighbouring positions carry nearly the same depth: one copy would make
    // most lanes of a warp meet on one counter), 8 words apart in their banks; summed into the first copy afterwards
    constexpr int kFineStride = 264;
    __shared__ __align__(16) u32 fine[4 * kFineStride];
    __shared__ u32 sel[4];                                   // per median: coarse bin (or 0xffffffff / 0xfffffffe = none / done), remainder or value
    __shared__ u32 s_list, s_val;
    const int c = blockIdx.x, t = threadIdx.x, lane = t & 31;
    const uint16_t *cov = planes + ((size_t)c * MGATK_N_PLANES + MGATK_PLANE_COVERAGE) * ppad;
    hist[t] = 0;
    for (int e = t; e < 4 * kFineStride; e += 256) fine[e] = 0;
    if (t == 0) s_list = 0;
    __syncthreads();
    {   // eight positions per load (rows are 128-byte aligned, the padding beyond P is zero)
        const uint4 *row = reinterpret_cast<const uint4 *>(cov);
        u32 *mine = fine + (lane & 3) * kFineStride;
        for (int q = t; q < ppad / 8; q += 256) {
            const uint4 w = __ldg(row + q);
            const u32 x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const u32 a = x[k] & 0xffffu, b = x[k] >> 16;
                if (a) atomicAdd(a < 256u ? &mine[a] : &hist[a >> 8], 1u);
                if (b) atomicAdd(b < 256u ? &mine[b] : &hist[b >> 8], 1u);
            }
        }
    }
    // saturated positions of this cell whose exact depth sits in the overflow list
    const bool deep = qc[c].max_depth > 65535u && ovf != nullptr;
    const int64_t n_list = deep ? min((int64_t)stats->n_overflow, ovf_cap) : 0;
    const u32 want = ((u32)MGATK_PLANE_COVERAGE << 24);
    if (deep) {
        u32 mine = 0;
        for (int64_t e = t; e < n_list; e += 256) mine += ovf[e].cell == c && (ovf[e].plane_pos & 0xff000000u) == want;
        if (mine) atomicAdd(&s_list, mine);
    }
    __syncthreads();
    fine[t] += fine[kFineStride + t] + fine[2 * kFineStride + t] + fine[3 * kFineStride + t];      // (thread t alone touches bin t)
    __syncthreads();
    if (t < 32) {                                            // warp 0: totals and both selections
        u32 bin, n_low, n_high, dummy;
        median_scan_warp(fine, 0u, bin, n_low, lane);
        median_scan_warp(hist, 0u, bin, n_high, lane);
        const u32 n = n_low + n_high;
        for (int s = 0; s < 2; s++) {
            const u32 k = s == 0 ? (n - 1) / 2 : n / 2;
            u32 b = 0xffffffffu, r = 0;
            if (n) {
                if (k < n_low) { median_scan_warp(fine, k, r, dummy, lane); b = 0xfffffffeu; }       // the depth itself
                else r = median_scan_warp(hist, k - n_low, b, dummy, lane);
            }
            if (lane == 0) { sel[2 * s] = b; sel[2 * s + 1] = r; }
        }
        if (lane == 0) s_val = n;
    }
    __syncthreads();
    if (sel[0] == 0xffffffffu) { if (t == 0) { qc[c].median_lo = 0; qc[c].median_hi = 0; } return; }
    const u32 n = s_val, n_below = n - s_list;               // values below the listed ones (a true 65535 included)
    const u32 k[2] = {(n - 1) / 2, n / 2};
    u32 res[2] = {0, 0};
    bool have_low = false;                                   // hist holds the low-byte histogram of bin sel[0]
    for (int s = 0; s < 2; s++) {
        if (k[s] >= n_below) {                               // the (k - n_below)-th smallest listed depth
            u32 rem = k[s] - n_below, prefix = 0, mask = 0;
            for (int shift = 24; shift >= 0; shift -= 8) {
                __syncthreads();
                hist[t] = 0;
                __syncthreads();
                for (int64_t e = t; e < n_list; e += 256)
                    if (ovf[e].cell == c && (ovf[e].plane_pos & 0xff000000u) == want && (ovf[e].value & mask) == prefix)
                        atomicAdd(&hist[(ovf[e].value >> shift) & 255u], 1u);
                __syncthreads();
                if (t == 0) { u32 bin; const u32 r = median_scan(hist, rem, bin); sel[0] = bin; sel[1] = r; }
                __syncthreads();
                prefix |= sel[0] << shift; mask |= 255u << shift; rem = sel[1];
            }
            res[s] = prefix;
            continue;
        }
        const u32 bin = sel[2 * s], rem = sel[2 * s + 1];
        if (bin == 0xfffffffeu) { res[s] = rem; continue; }   // below 256: read off the exact histogram
        if (!(s == 1 && have_low && bin == sel[0])) {        // (same high byte as the lower median: its low-byte histogram is still valid)
            __syncthreads();
            hist[t] = 0;
            __syncthreads();
            const uint4 *row = reinterpret_cast<const uint4 *>(cov);
            for (int q = t; q < ppad / 8; q += 256) {
                const uint4 w = __ldg(row + q);
                const u32 x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int kk = 0; kk < 4; kk++) {
                    const u32 a = x[kk] & 0xffffu, b = x[kk] >> 16;
                    if (a && (a >> 8) == bin) atomicAdd(&hist[a & 255u], 1u);
                    if (b && (b >> 8) == bin) atomicAdd(&hist[b & 255u], 1u);
                }
            }
            __syncthreads();
            have_low = s == 0;
        }
        if (t == 0) { u32 b; median_scan(hist, rem, b); s_val = (bin << 8) | b; }
        __syncthreads();
        res[s] = s_val;
    }
    if (t == 0) { qc[c].median_lo = res[0]; qc[c].median_hi = res[1]; }
}
#else
__global__ void __launch_bounds__(256)
k_median(const uint16_t *__restrict__ planes, int P, int ppad, mgatk_cell_qc *__restrict__ qc,
         const mgatk_overflow *__restrict__ ovf, const mgatk_stats *__restrict__ stats, int64_t ovf_cap,
         const u32 *__restrict__ t32, u64 *__restrict__ totals) {
    if (t32)                                                 // the base totals the pileup kernel reduced, widened to int64 [P][4] (k_totals_widen)
        for (int p = blockIdx.x * 256 + threadIdx.x; p < P; p += gridDim.x * 256) {
            ulonglong2 lo, hi;
            lo.x = t32[p]; lo.y = t32[(size_t)ppad + p]; hi.x = t32[(size_t)2 * ppad + p]; hi.y = t32[(size_t)3 * ppad + p];
            reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p] = lo;
            reinterpret_cast<ulonglong2 *>(totals)[2 * (size_t)p + 1] = hi;
        }
    __shared__ u32 hist[256];
    __shared__ u32 sel[4];                                   // bin, remainder for lo / hi
    __shared__ u32 s_list, s_val;
    const int c = blockIdx.x, t = threadIdx.x;
    const uint16_t *cov = planes + ((size_t)c * MGATK_N_PLANES + MGATK_PLANE_COVERAGE) * ppad;
    hist[t] = 0;
    if (t == 0) s_list = 0;
    __syncthreads();
    {   // eight positions per load (rows are 128-byte aligned, the padding beyond P is zero); depths below 256 - nearly
        // all of them - are counted in a register instead of hammering one shared counter
        u32 low = 0;
        const uint4 *row = reinterpret_cast<const uint4 *>(cov);
        for (int q = t; q < ppad / 8; q += 256) {
            const uint4 w = __ldg(row + q);
            const u32 x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const u32 a = x[k] & 0xffffu, b = x[k] >> 16;
                if (a) { if (a < 256u) low++; else atomicAdd(&hist[a >> 8], 1u); }
                if (b) { if (b < 256u) low++; else atomicAdd(&hist[b >> 8], 1u); }
            }
        }
        low = __reduce_add_sync(kFull, low);
        if ((t & 31) == 0 && low) atomicAdd(&hist[0], low);
    }
    // saturated positions of this cell whose exact depth sits in the overflow list
    const bool deep = qc[c].max_depth > 65535u && ovf != nullptr;
    const int64_t n_list = deep ? min((int64_t)stats->n_overflow, ovf_cap) : 0;
    const u32 want = ((u32)MGATK_PLANE_COVERAGE << 24);
    if (deep) {
        u32 mine = 0;
        for (int64_t e = t; e < n_list; e += 256) mine += ovf[e].cell == c && (ovf[e].plane_pos & 0xff000000u) == want;
        if (mine) atomicAdd(&s_list, mine);
    }
    __syncthreads();
    u32 res[2] = {0, 0};
    u32 k[2] = {0, 0}, n_below = 0;
    if (t == 0) {
        u32 n = 0;
        for (int b = 0; b < 256; b++) n += hist[b];
        sel[0] = sel[2] = 0xffffffffu;
        if (n) {
            k[0] = (n - 1) / 2; k[1] = n / 2;
            for (int s = 0; s < 2; s++) sel[2 * s + 1] = median_scan(hist, k[s], sel[2 * s]);
        }
        s_val = n;
    }
    __syncthreads();
    if (sel[0] == 0xffffffffu) { if (t == 0) { qc[c].median_lo = 0; qc[c].median_hi = 0; } return; }
    {
        const u32 n = s_val;
        k[0] = (n - 1) / 2; k[1] = n / 2;
        n_below = n - s_list;                                // values below the listed ones (a true 65535 included)
    }
    for (int s = 0; s < 2; s++) {
        if (k[s] >= n_below) {                               // the (k - n_below)-th smallest listed depth
            u32 rem = k[s] - n_below, prefix = 0, mask = 0;
            for (int shift = 24; shift >= 0; shift -= 8) {
                __syncthreads();
                hist[t] = 0;
                __syncthreads();
                for (int64_t e = t; e < n_list; e += 256)
                    if (ovf[e].cell == c && (ovf[e].plane_pos & 0xff000000u) == want && (ovf[e].value & mask) == prefix)
                        atomicAdd(&hist[(ovf[e].value >> shift) & 255u], 1u);
                __syncthreads();
                if (t == 0) { u32 bin; const u32 r = median_scan(hist, rem, bin); sel[0] = bin; sel[1] = r; }
                __syncthreads();
                prefix |= sel[0] << shift; mask |= 255u << shift; rem = sel[1];
            }
            res[s] = prefix;
            continue;
        }
        const u32 bin = sel[2 * s], rem = sel[2 * s + 1];
        if (!(s == 1 && bin == sel[0])) {                    // (same high byte as the lower median: its low-byte histogram is still valid)
            __syncthreads();
            hist[t] = 0;
            __syncthreads();
            const uint4 *row = reinterpret_cast<const uint4 *>(cov);
            for (int q = t; q < ppad / 8; q += 256) {
                const uint4 w = __ldg(row + q);
                const u32 x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const u32 a = x[k] & 0xffffu, b = x[k] >> 16;
                    if (a && (a >> 8) == bin) atomicAdd(&hist[a & 255u], 1u);
                    if (b && (b >> 8) == bin) atomicAdd(&hist[b & 255u], 1u);
                }
            }
            __syncthreads();
        }
        if (t == 0) { u32 b; median_scan(hist, rem, b); s_val = (bin << 8) | b; }
        __syncthreads();
        res[s] = s_val;
    }
    if (t == 0) { qc[c].median_lo = res[0]; qc[c].median_hi = res[1]; }
}
#endif

}  // namespace mgatk
