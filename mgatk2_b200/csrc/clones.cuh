// mgatk2_b200 — clones (include/mgatk2_b200.h, mgatk_clone_*; DESIGN §8 "Clones").
//
// The second half of the Signac clone workflow, after the variant call: heteroplasmy x[c, v] = (f + r) / d of the called
// variants (AlleleFreq), the exact cosine k nearest neighbours of the graph rows, the shared-nearest-neighbour weights of
// the kNN edges, and deterministic Louvain on the host.
//
//   * k_clone_af builds x (row-major [n][vpad], zero beyond V) and inv[i] = 1 / sqrt(dot(i, i)) in handle scratch (0 for
//     an all-zero row, so every cosine is a number and the order stays total);
//   * k_clone_knn: one CTA owns kCloneTile query rows and walks every candidate tile of kCloneTile rows in ascending
//     order. The dot products of the tile pair are accumulated in a 4 x 4 register micro-tile per thread from x stages of
//     kCloneVC variants in shared memory, v ascending, one rounded multiply and one rounded add per term (no FMA), so each
//     dot has the bits of the sequential sum. Each query row keeps its best k_eff - 1 others sorted by (cos desc, index
//     asc) in shared memory; a candidate that does not beat the row's current last entry is rejected in registers, the
//     survivors are merged by rank (one warp per row). The n x n matrix is never written;
//   * k_clone_snn: one warp per row counts |N(i) ∩ N(j)| for every j of N(i) against a sorted copy of N(i).
#pragma once
#include "common.cuh"

#include <algorithm>
#include <cmath>
#include <new>
#include <vector>

namespace mgatk {

constexpr int kCloneKMax = 64;          // MGATK_CLONE_K_MAX
constexpr int kCloneTile = 64;          // query rows per CTA = candidate rows per step
constexpr int kCloneVC = 32;            // variants per shared-memory stage; x rows are padded to a multiple of it
constexpr int kCloneThreads = 256;      // 16 x 16 threads, 4 x 4 pairs each
constexpr int kClonePitch = kCloneTile + 1;

__host__ __device__ inline int clone_vpad(int V) { return (V + kCloneVC - 1) / kCloneVC * kCloneVC; }

// x = (f + r) / d of cell c in variant v, 0 when d = 0; counts is [V][3][C] of mgatk_variant_cells_device (also the x of
// the marker ranks, markers.cuh)
__device__ __forceinline__ double allele_frequency(const u32 *counts, int C, int v, int c) {
    const u32 *cv = counts + (size_t)3 * v * C + c;
    const u32 d = cv[2 * (size_t)C];
    return d ? __ddiv_rn((double)((u64)cv[0] + cv[C]), (double)d) : 0.0;
}

// x[i][v] and inv[i] of graph row i (cell rows[i]); counts is [V][3][C] of mgatk_variant_cells_device
__global__ void k_clone_af(const u32 *counts, const int32_t *rows, int n, int C, int V, int vpad, double *x, double *inv) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = rows[i];
    const bool ok = c >= 0 && c < C;
    double acc = 0.0;
    for (int v = 0; v < vpad; v++) {
        const double xv = ok && v < V ? allele_frequency(counts, C, v, c) : 0.0;
        x[(size_t)i * vpad + v] = xv;
        acc = __dadd_rn(acc, __dmul_rn(xv, xv));
    }
    inv[i] = acc > 0.0 ? __ddiv_rn(1.0, __dsqrt_rn(acc)) : 0.0;     // a row without a detection: every cosine 0, never NaN
}

struct CloneKnnSmem {
    union {
        struct { double q[kCloneVC][kClonePitch], c[kCloneVC][kClonePitch]; } x;   // x stages, transposed
        double cos[kCloneTile][kClonePitch];                                        // survivors of one tile pair
    } u;
    double lsim[kCloneTile][kCloneKMax];        // per query row: its best others, (cos desc, index asc)
    int lidx[kCloneTile][kCloneKMax];
    unsigned long long cand[kCloneTile];        // survivor columns of the current candidate tile
    int lcount[kCloneTile];
};

// (s1, j1) comes before (s2, j2): larger cosine, on a tie the lower row
__device__ __forceinline__ bool knn_before(double s1, int j1, double s2, int j2) { return s1 > s2 || (s1 == s2 && j1 < j2); }

__global__ void __launch_bounds__(kCloneThreads, 2)
k_clone_knn(const double *__restrict__ x, const double *__restrict__ inv, int n, int vpad, int k_eff,
            int32_t *nbr_out, double *sim_out) {
    extern __shared__ __align__(16) unsigned char clone_smem[];
    CloneKnnSmem &sm = *reinterpret_cast<CloneKnnSmem *>(clone_smem);
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4, lane = tid & 31, warp = tid >> 5;
    const int q0 = blockIdx.x * kCloneTile;
    const int kp = k_eff - 1;                   // others per row, >= 1
    if (tid < kCloneTile) { sm.cand[tid] = 0; sm.lcount[tid] = 0; }
    double inv_q[4];
#pragma unroll
    for (int a = 0; a < 4; a++) {
        const int i = q0 + ty + 16 * a;
        inv_q[a] = i < n ? inv[i] : 0.0;
    }

    for (int c0 = 0; c0 < n; c0 += kCloneTile) {
        double acc[4][4];
#pragma unroll
        for (int a = 0; a < 4; a++)
#pragma unroll
            for (int b = 0; b < 4; b++) acc[a][b] = 0.0;
        for (int v0 = 0; v0 < vpad; v0 += kCloneVC) {
            __syncthreads();                    // the union is free: last stage read, last merge done
            for (int e = tid; e < kCloneTile * kCloneVC; e += kCloneThreads) {
                const int r = e / kCloneVC, v = e % kCloneVC;
                const int qi = q0 + r, ci = c0 + r;
                sm.u.x.q[v][r] = qi < n ? x[(size_t)qi * vpad + v0 + v] : 0.0;
                sm.u.x.c[v][r] = ci < n ? x[(size_t)ci * vpad + v0 + v] : 0.0;
            }
            __syncthreads();
#pragma unroll 8
            for (int v = 0; v < kCloneVC; v++) {
                double qa[4], cb[4];
#pragma unroll
                for (int a = 0; a < 4; a++) qa[a] = sm.u.x.q[v][ty + 16 * a];
#pragma unroll
                for (int b = 0; b < 4; b++) cb[b] = sm.u.x.c[v][tx + 16 * b];
#pragma unroll
                for (int a = 0; a < 4; a++)
#pragma unroll
                    for (int b = 0; b < 4; b++) acc[a][b] = __dadd_rn(acc[a][b], __dmul_rn(qa[a], cb[b]));
            }
        }
        __syncthreads();                        // x stages read: the union becomes the survivor tile

        // ---- cosines, rejected against each row's current last entry ----
        double inv_c[4];
#pragma unroll
        for (int b = 0; b < 4; b++) {
            const int j = c0 + tx + 16 * b;
            inv_c[b] = j < n ? inv[j] : 0.0;
        }
#pragma unroll
        for (int a = 0; a < 4; a++) {
            const int r = ty + 16 * a, i = q0 + r;
            if (i >= n) continue;
            const bool full = sm.lcount[r] == kp;
            const double ts = full ? sm.lsim[r][kp - 1] : 0.0;
            const int ti = full ? sm.lidx[r][kp - 1] : 0;
            unsigned long long bits = 0;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int col = tx + 16 * b, j = c0 + col;
                if (j >= n || j == i) continue;
                const double s = __dmul_rn(__dmul_rn(acc[a][b], inv_q[a]), inv_c[b]);
                if (!full || knn_before(s, j, ts, ti)) {
                    sm.u.cos[r][col] = s;
                    bits |= 1ull << col;
                }
            }
            if (bits) atomicOr(&sm.cand[r], bits);
        }
        __syncthreads();

        // ---- merge the survivors of each row into its list: one warp per row, by rank in the union ----
        for (int r = warp; r < kCloneTile; r += kCloneThreads / 32) {
            const unsigned long long m = sm.cand[r];
            if (!m) continue;
            const int L = sm.lcount[r];
            double es[4];
            int ej[4], rank[4];
#pragma unroll
            for (int t = 0; t < 4; t++) {           // t 0, 1: list entries lane, lane + 32; t 2, 3: columns lane, lane + 32
                const int e = lane + 32 * (t & 1);
                rank[t] = kCloneKMax;               // not an element
                if (t < 2) {
                    if (e >= L) continue;
                    es[t] = sm.lsim[r][e]; ej[t] = sm.lidx[r][e];
                    rank[t] = e;                    // the list is sorted and its entries are distinct
                } else {
                    if (!((m >> e) & 1)) continue;
                    es[t] = sm.u.cos[r][e]; ej[t] = c0 + e;
                    int rk = 0;
                    for (int l = 0; l < L; l++) rk += knn_before(sm.lsim[r][l], sm.lidx[r][l], es[t], ej[t]);
                    rank[t] = rk;
                }
                for (unsigned long long mm = m; mm; mm &= mm - 1) {
                    const int col = __ffsll((long long)mm) - 1;
                    rank[t] += knn_before(sm.u.cos[r][col], c0 + col, es[t], ej[t]);
                }
            }
            __syncwarp();
#pragma unroll
            for (int t = 0; t < 4; t++)
                if (rank[t] < kp) { sm.lsim[r][rank[t]] = es[t]; sm.lidx[r][rank[t]] = ej[t]; }
            __syncwarp();
            if (lane == 0) {
                const int T = L + __popcll(m);
                sm.lcount[r] = T < kp ? T : kp;
                sm.cand[r] = 0;
            }
        }
    }
    __syncthreads();

    // ---- N(i): i itself with 1.0, then the list ----
    for (int e = tid; e < kCloneTile * k_eff; e += kCloneThreads) {
        const int r = e / k_eff, t = e % k_eff, i = q0 + r;
        if (i >= n) continue;
        nbr_out[(size_t)i * k_eff + t] = t == 0 ? i : sm.lidx[r][t - 1];
        sim_out[(size_t)i * k_eff + t] = t == 0 ? 1.0 : sm.lsim[r][t - 1];
    }
}

// N(i) of a row with only itself (n = 1)
__global__ void k_clone_self(int n, int k_eff, int32_t *nbr_out, double *sim_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { nbr_out[(size_t)i * k_eff] = i; sim_out[(size_t)i * k_eff] = 1.0; }
}

constexpr int kSnnWarps = 8;

// w[i][t] = s / (2 k - s), s = |N(i) ∩ N(nbr[i][t])|; one warp per row
__global__ void __launch_bounds__(kSnnWarps * 32) k_clone_snn(const int32_t *nbr, int n, int k, double *w) {
    __shared__ int sorted[kSnnWarps][kCloneKMax];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = blockIdx.x * kSnnWarps + warp;
    if (i >= n) return;                         // whole warps leave; no CTA barrier follows
    const int32_t *ni = nbr + (size_t)i * k;
    const int e0 = lane < k ? ni[lane] : INT32_MAX, e1 = lane + 32 < k ? ni[lane + 32] : INT32_MAX;
    int r0 = 0, r1 = 0;                         // rank sort: the entries of a row are distinct
    for (int t = 0; t < k; t++) {
        const int a = __shfl_sync(0xffffffffu, e0, t & 31), b = __shfl_sync(0xffffffffu, e1, t & 31);
        const int v = t < 32 ? a : b;
        r0 += v < e0; r1 += v < e1;
    }
    if (lane < k) sorted[warp][r0] = e0;
    if (lane + 32 < k) sorted[warp][r1] = e1;
    __syncwarp();
    for (int t = 0; t < k; t++) {
        const int j = ni[t];
        int s = 0;
        if (j >= 0 && j < n) {
            const int32_t *nj = nbr + (size_t)j * k;
            bool hit[2] = {false, false};
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int e = lane + 32 * h;
                if (e >= k) continue;
                const int val = nj[e];
                int lo = 0, hi = k;             // first sorted entry >= val
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (sorted[warp][mid] < val) lo = mid + 1; else hi = mid;
                }
                hit[h] = lo < k && sorted[warp][lo] == val;
            }
            s = __popc(__ballot_sync(0xffffffffu, hit[0])) + __popc(__ballot_sync(0xffffffffu, hit[1]));
        }
        if (lane == 0) w[(size_t)i * k + t] = __ddiv_rn((double)s, (double)(2 * k - s));
    }
}

// ---------------------------------------------------------------------------------------------
// deterministic Louvain (host). Every float operation below is a plain IEEE fp64 add, multiply or divide in the order
// DESIGN §8 "Clones" states, so oracle/clones.py reproduces the labels; no expression has the shape a * b + c.
// ---------------------------------------------------------------------------------------------
struct LouvainGraph {
    std::vector<int64_t> indptr;
    std::vector<int32_t> indices;
    std::vector<double> weights;
};

// phase 1 on g; comm[i] in, moved nodes' communities out. Returns whether any node moved.
inline bool louvain_phase1(const LouvainGraph &g, double resolution, std::vector<int32_t> &comm) {
    const int n = (int)g.indptr.size() - 1;
    std::vector<double> k(n, 0.0), tot(n, 0.0);
    double m2 = 0.0;
    for (int i = 0; i < n; i++) {
        double s = 0.0;
        for (int64_t e = g.indptr[i]; e < g.indptr[i + 1]; e++) s = s + g.weights[e];
        k[i] = s;
        m2 = m2 + s;
    }
    for (int i = 0; i < n; i++) tot[comm[i]] = tot[comm[i]] + k[i];
    if (!(m2 > 0.0)) return false;
    std::vector<double> wc(n, 0.0);
    std::vector<int32_t> seen, stamp(n, -1);       // communities next to i (stamp[c] == i), in first-seen order
    bool any = false;
    for (int sweep = 0; sweep < 100; sweep++) {
        bool moved = false;
        for (int i = 0; i < n; i++) {
            const int32_t old = comm[i];
            const double tot_old = tot[old];
            tot[old] = tot_old - k[i];                     // i isolated
            seen.clear();
            seen.push_back(old);
            stamp[old] = i;
            wc[old] = 0.0;
            for (int64_t e = g.indptr[i]; e < g.indptr[i + 1]; e++) {
                const int32_t j = g.indices[e];
                if (j == i) continue;
                const int32_t c = comm[j];
                if (stamp[c] != i) { stamp[c] = i; seen.push_back(c); wc[c] = 0.0; }
                wc[c] = wc[c] + g.weights[e];
            }
            auto gain = [&](int32_t c) {
                double t = tot[c] * k[i];
                t = resolution * t;
                t = t / m2;
                return wc[c] - t;
            };
            const double own = gain(old);
            int32_t best = old;
            double best_gain = own;
            for (int32_t c : seen) {
                const double gc = gain(c);
                if (gc > best_gain || (gc == best_gain && c < best)) { best = c; best_gain = gc; }
            }
            if (best != old && best_gain > own) {
                comm[i] = best;
                tot[best] = tot[best] + k[i];
                moved = true;
            } else {
                tot[old] = tot_old;
            }
        }
        if (!moved) break;
        any = true;
    }
    return any;
}

// labels[i] in 1..K for a CSR graph (see mgatk_louvain_host)
inline void louvain(LouvainGraph g, double resolution, int32_t *labels, int32_t *n_levels) {
    const int n0 = (int)g.indptr.size() - 1;
    std::vector<int32_t> node_of(n0);              // original node -> node of the current level
    for (int i = 0; i < n0; i++) node_of[i] = i;
    int levels = 0;
    for (;;) {
        const int n = (int)g.indptr.size() - 1;
        std::vector<int32_t> comm(n);
        for (int i = 0; i < n; i++) comm[i] = i;
        if (!louvain_phase1(g, resolution, comm)) break;
        levels++;
        // community index = rank of its smallest member
        std::vector<int32_t> first(n, -1), id(n, -1);
        for (int i = 0; i < n; i++) if (first[comm[i]] < 0) first[comm[i]] = i;
        int nc = 0;
        for (int i = 0; i < n; i++) if (first[comm[i]] == i) id[comm[i]] = nc++;
        for (int i = 0; i < n0; i++) node_of[i] = id[comm[node_of[i]]];
        // aggregate: A'[C][D] sums A[i][j] in (i asc, j asc) order
        struct E { int32_t c, d; int64_t order; double w; };
        std::vector<E> es;
        es.reserve(g.indices.size());
        for (int i = 0; i < n; i++)
            for (int64_t e = g.indptr[i]; e < g.indptr[i + 1]; e++) es.push_back({id[comm[i]], id[comm[g.indices[e]]], e, g.weights[e]});
        std::sort(es.begin(), es.end(), [](const E &a, const E &b) {
            return a.c != b.c ? a.c < b.c : a.d != b.d ? a.d < b.d : a.order < b.order;
        });
        LouvainGraph h;
        h.indptr.assign(nc + 1, 0);
        for (size_t s = 0; s < es.size();) {
            size_t t = s;
            double w = 0.0;
            for (; t < es.size() && es[t].c == es[s].c && es[t].d == es[s].d; t++) w = w + es[t].w;
            h.indices.push_back(es[s].d);
            h.weights.push_back(w);
            h.indptr[es[s].c + 1]++;
            s = t;
        }
        for (int c = 0; c < nc; c++) h.indptr[c + 1] += h.indptr[c];
        g = std::move(h);
    }
    // clone numbers: size descending, ties to the smallest member
    const int n = (int)g.indptr.size() - 1;
    std::vector<int64_t> size(n, 0);
    std::vector<int32_t> first(n, -1);
    for (int i = 0; i < n0; i++) { size[node_of[i]]++; if (first[node_of[i]] < 0) first[node_of[i]] = i; }
    std::vector<int32_t> order(n);
    for (int c = 0; c < n; c++) order[c] = c;
    std::sort(order.begin(), order.end(), [&](int32_t a, int32_t b) {
        return size[a] != size[b] ? size[a] > size[b] : first[a] < first[b];
    });
    std::vector<int32_t> number(n);
    for (int r = 0; r < n; r++) number[order[r]] = r + 1;
    for (int i = 0; i < n0; i++) labels[i] = number[node_of[i]];
    *n_levels = levels;
}

}  // namespace mgatk
