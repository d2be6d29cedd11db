// mgatk2_b200 — clone markers (include/mgatk2_b200.h, mgatk_marker_ranks_device; DESIGN §8 "Clone markers").
//
// Wilcoxon rank sums of x = (f + r) / d per variant, each group against the rest: the exact integers
// rank2[v][g] = sum over the group's cells of 2 * mid-rank and ties[v] = sum over runs of equal x of t^3 - t, from which
// the host forms U, the tie-corrected normal approximation and p (markers.py).
//
//   * k_marker_split, one thread per (cell, variant): x by allele_frequency (clones.cuh, the x of k_clone_af); the
//     nonzero (bits of x, label) pairs of the population are compacted into handle scratch at variant v's slots
//     [v * C, v * C + nnz[v]), reserved with one atomic per warp. The row of variant 0 also counts the group sizes and
//     the population N. The order inside the scratch is not deterministic; only integer sums leave the kernels.
//   * k_marker_rank, one CTA per variant (grid-strided): the zeros are never sorted. The nonzero x are positive doubles
//     <= 1, so their bit patterns sort as unsigned integers. Up to kMarkerS of them are sorted in shared memory (bitonic);
//     more take the fallback: chunks of kMarkerS sorted in shared memory, then merge passes through global ping-pong
//     scratch of the CTA (each element's place found by binary search in the partner run). In the sorted nonzeros an
//     element with lo = first index of its value and hi = one past the last has mid-rank z + (lo + hi + 1) / 2 among
//     the population (z = N - nnz zeros ranked first), so it adds z + lo + hi to its group (the group's zeros and its
//     nonzeros' other z + 1 are added once as n_g * (z + 1)) and (hi - lo)^2 - 1 to ties (a run of t adds t^3 - t).
//     Group sums go to shared memory when G <= kMarkerGs, else straight to the output with u64 atomics.
#pragma once
#include "common.cuh"
#include "clones.cuh"

namespace mgatk {

constexpr int kMarkerS = 4096;          // nonzero values sorted in shared memory; more take the global merge fallback
constexpr int kMarkerGs = 1024;         // groups accumulated in shared memory; more add to the output directly
constexpr int kMarkerThreads = 512;
constexpr int kMarkerSplitThreads = 256;

struct MarkerSmem {
    u64 key[kMarkerS];
    int32_t lab[kMarkerS];
    u64 acc[kMarkerGs];
    u64 ties;
};

// counters: nnz [V], group sizes [G + 1] (index = label), N [1]; all zero on entry
__global__ void __launch_bounds__(kMarkerSplitThreads)
k_marker_split(const u32 *counts, const int32_t *labels, int C, int G, u32 *nnz, u32 *gsize, u32 *npop, u64 *keys,
               int32_t *labs) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x, v = blockIdx.y, lane = threadIdx.x & 31;
    const int g = c < C ? labels[c] : 0;
    const bool in = g >= 1 && g <= G;
    const double x = in ? allele_frequency(counts, C, v, c) : 0.0;
    const bool hit = x > 0.0;
    const u32 m = __ballot_sync(kFull, hit);
    if (m) {
        const int leader = __ffs(m) - 1;
        u32 base = 0;
        if (lane == leader) base = atomicAdd(&nnz[v], (u32)__popc(m));
        base = __shfl_sync(kFull, base, leader);
        if (hit) {
            const size_t slot = (size_t)v * C + base + __popc(m & ((1u << lane) - 1));
            keys[slot] = (u64)__double_as_longlong(x);
            labs[slot] = g;
        }
    }
    if (v == 0) {
        const u32 mi = __ballot_sync(kFull, in);
        if (lane == 0 && mi) atomicAdd(npop, (u32)__popc(mi));
        if (in) {
            const u32 peers = __match_any_sync(mi, g);
            if (lane == __ffs(peers) - 1) atomicAdd(&gsize[g], (u32)__popc(peers));
        }
    }
}

// first index in [lo, hi) whose key is >= x (kUpper: > x), hi when there is none
template <bool kUpper>
__device__ __forceinline__ int marker_bound(const u64 *key, int lo, int hi, u64 x) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (kUpper ? key[mid] <= x : key[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// ascending bitonic sort of (key, lab)[0, n2), n2 a power of two <= kMarkerS; the caller has synchronised after filling
__device__ void marker_sort_smem(u64 *key, int32_t *lab, int n2) {
    for (int k = 2; k <= n2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n2; i += blockDim.x) {
                const int l = i ^ j;
                if (l > i) {
                    const u64 a = key[i], b = key[l];
                    if ((a > b) == ((i & k) == 0)) {
                        key[i] = b; key[l] = a;
                        const int32_t t = lab[i]; lab[i] = lab[l]; lab[l] = t;
                    }
                }
            }
            __syncthreads();
        }
}

// the sorted nonzeros key[0, n) of one variant: z + lo + hi to each element's group, the sum of (hi - lo)^2 - 1 returned
__device__ u64 marker_score(const u64 *key, const int32_t *lab, int n, u64 z, bool shared_acc, u64 *acc, u64 *r2) {
    u64 tie = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const u64 x = key[i];
        const int lo = marker_bound<false>(key, 0, i, x), hi = marker_bound<true>(key, i + 1, n, x);
        const u64 t = (u64)(hi - lo);
        tie += t * t - 1;
        const u64 c = z + (u64)lo + (u64)hi;
        const int g = lab[i] - 1;
        atomicAdd(shared_acc ? &acc[g] : &r2[g], c);
    }
    return tie;
}

// keys / labs: [V][C] of k_marker_split (overwritten by the fallback); tkeys / tlabs: [gridDim.x][C] ping-pong scratch
// of the fallback (unused when C <= kMarkerS)
__global__ void __launch_bounds__(kMarkerThreads)
k_marker_rank(u64 *keys, int32_t *labs, const u32 *nnz, const u32 *gsize, const u32 *npop, int C, int V, int G,
              u64 *tkeys, int32_t *tlabs, u64 *rank2, u64 *ties_out) {
    extern __shared__ __align__(16) unsigned char marker_smem[];
    MarkerSmem &sm = *reinterpret_cast<MarkerSmem *>(marker_smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const bool shared_acc = G <= kMarkerGs;
    const u64 N = *npop;
    for (int v = blockIdx.x; v < V; v += gridDim.x) {
        const int n = (int)nnz[v];
        const u64 z = N - (u64)n;
        u64 *r2 = rank2 + (size_t)v * G;
        u64 *ka = keys + (size_t)v * C;
        int32_t *la = labs + (size_t)v * C;
        __syncthreads();                        // shared memory of the previous variant read
        if (tid == 0) sm.ties = 0;
        for (int g = tid; g < G; g += blockDim.x) {
            if (shared_acc) sm.acc[g] = 0;
            else r2[g] = (u64)gsize[g + 1] * (z + 1);
        }
        u64 tie = 0;
        if (n <= kMarkerS) {
            int n2 = 1;
            while (n2 < n) n2 <<= 1;
            for (int i = tid; i < n2; i += blockDim.x) {
                sm.key[i] = i < n ? ka[i] : ~0ull;
                sm.lab[i] = i < n ? la[i] : 0;
            }
            __syncthreads();
            marker_sort_smem(sm.key, sm.lab, n2);
            tie = marker_score(sm.key, sm.lab, n, z, shared_acc, sm.acc, r2);
        } else {
            for (int c0 = 0; c0 < n; c0 += kMarkerS) {
                const int m = n - c0 < kMarkerS ? n - c0 : kMarkerS;
                __syncthreads();                // the previous chunk is written back
                for (int i = tid; i < kMarkerS; i += blockDim.x) {
                    sm.key[i] = i < m ? ka[c0 + i] : ~0ull;
                    sm.lab[i] = i < m ? la[c0 + i] : 0;
                }
                __syncthreads();
                marker_sort_smem(sm.key, sm.lab, kMarkerS);
                for (int i = tid; i < m; i += blockDim.x) { ka[c0 + i] = sm.key[i]; la[c0 + i] = sm.lab[i]; }
            }
            __syncthreads();
            u64 *kb = tkeys + (size_t)blockIdx.x * C;
            int32_t *lb = tlabs + (size_t)blockIdx.x * C;
            for (int w = kMarkerS; w < n; w <<= 1) {
                for (int i = tid; i < n; i += blockDim.x) {
                    const int start = i / (2 * w) * (2 * w);
                    const int mid = start + w < n ? start + w : n, end = start + 2 * w < n ? start + 2 * w : n;
                    const u64 x = ka[i];
                    const int pos = i < mid ? (i - start) + (marker_bound<false>(ka, mid, end, x) - mid)
                                            : (i - mid) + (marker_bound<true>(ka, start, mid, x) - start);
                    kb[start + pos] = x;
                    lb[start + pos] = la[i];
                }
                __syncthreads();
                u64 *tk = ka; ka = kb; kb = tk;
                int32_t *tl = la; la = lb; lb = tl;
            }
            tie = marker_score(ka, la, n, z, shared_acc, sm.acc, r2);
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) tie += __shfl_down_sync(kFull, tie, o);
        if (lane == 0) atomicAdd(&sm.ties, tie);
        __syncthreads();
        if (shared_acc)
            for (int g = tid; g < G; g += blockDim.x) r2[g] = (u64)gsize[g + 1] * (z + 1) + sm.acc[g];
        if (tid == 0) ties_out[v] = sm.ties + z * z * z - z;
    }
}

}  // namespace mgatk
