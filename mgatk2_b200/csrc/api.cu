// mgatk2_b200 — C-ABI host side (include/mgatk2_b200.h). Launch sequencing, workspace carving,
// host-buffer entry point. No torch types; everything here is plain CUDA runtime.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "partition.cuh"
#include "dedup.cuh"
#include "pileup.cuh"
#include "epilogue.cuh"
#include "variants.cuh"
#include "clones.cuh"
#include "markers.cuh"
#include "deletions.cuh"

using namespace mgatk;

namespace {

constexpr int kMaxChunks = 148 * MGATK_SCATTER_CTAS * (256 / kPartThreads);   // partition CTAs: one wave (bounds the open write heads)
constexpr int kMaxDigitBits = 11;                    // 2048 bins * 20 B = 40 KB of shared memory per scatter CTA
constexpr int kMaxStages = 16;
constexpr int kTotalsMaxPpad = 1 << 16;              // contigs up to this long get their base totals from the pileup kernel itself

#ifndef MGATK_FUSED_SMALL
#define MGATK_FUSED_SMALL 1          // 1: bin totals by atomics + one-pass bin scan, stage1_reads published by k_find_long_runs, totals widened by k_median
#endif

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

int env_int(const char *name, int fallback) {
    const char *e = getenv(name);
    return e && *e ? atoi(e) : fallback;
}

struct Layout {          // carve-up of the caller's workspace
    int64_t n; int32_t n_cells;
    int nchunks; int64_t chunk; int ngroups;
    int passes, bits[2], shift[2];
    SlotFmt fmt;
    int stage_bytes, cap_reads, unit_reads; int64_t max_units;
    size_t slots[2];         // two slot arrays: partition output(s) and the compacted reads to pile up
    size_t mat, part, cell_start, cell_first, unit_start, units, units_big, scan_state, totals32, scalars, total;
    int64_t dedup_blocks;
};

// bytes of one stage of the main pileup kernel (= the slots of one unit) and the reads it holds
int stage_bytes_for(const SlotFmt &f) {
    int b = env_int("MGATK_STAGE_BYTES", f.compact ? 16384 : 32768);
    if (b < 32 * f.bytes) b = 32 * f.bytes;
    return (b + 127) / 128 * 128;
}

bool make_layout(int64_t n, int32_t n_cells, int extent, Layout &L) {
    if (n < 0 || n_cells < 0 || n >= (int64_t)0x7fffff00 || extent < 1) return false;
    L.n = n; L.n_cells = n_cells;
    int64_t nch = (n + 4095) / 4096;
    L.nchunks = (int)(nch < 1 ? 1 : nch > kMaxChunks ? kMaxChunks : nch);
    L.chunk = ((n + L.nchunks - 1) / L.nchunks + kPartThreads - 1) / kPartThreads * kPartThreads;
    if (L.chunk < kPartThreads) L.chunk = kPartThreads;
    L.ngroups = (L.nchunks + kScanGroup - 1) / kScanGroup;
    int bits = 1;
    while ((1ll << bits) < n_cells) bits++;
    if (bits > 2 * kMaxDigitBits) return false;
    L.passes = bits <= kMaxDigitBits ? 1 : 2;
    if (L.passes == 1) { L.bits[0] = bits; L.shift[0] = 0; L.bits[1] = 0; L.shift[1] = 0; }
    else { L.bits[0] = (bits + 1) / 2; L.shift[0] = 0; L.bits[1] = bits - L.bits[0]; L.shift[1] = L.bits[0]; }
    L.fmt = slot_format(extent);
    L.stage_bytes = stage_bytes_for(L.fmt);
    L.cap_reads = L.stage_bytes / L.fmt.bytes;
    {   // reads per unit: leave room for the reads of the halo and of the chunk the tile border is rounded down to
        const int v = env_int("MGATK_UNIT_READS", 0);
        L.unit_reads = v > 0 ? (v < 32 ? 32 : v) : (int)(0.68 * L.cap_reads);
        if (L.unit_reads < 32) L.unit_reads = 32;
    }
    L.max_units = (int64_t)n_cells + n / L.unit_reads + 1;
    const int max_bins = 1 << (L.bits[0] > L.bits[1] ? L.bits[0] : L.bits[1]);
    size_t o = 0;
    const size_t cap = (size_t)(n > 0 ? n : 1);
    for (int gen = 0; gen < 2; gen++) { L.slots[gen] = o; o += align_up(cap * (size_t)L.fmt.bytes); }
    L.mat = o; o += align_up((size_t)L.nchunks * max_bins * 4);
    L.part = o; o += align_up(((size_t)L.ngroups + 1) * max_bins * 4 + 4);      // group sums + one row of bin totals (+ their sum)
    L.cell_start = o; o += align_up(((size_t)n_cells + 1) * 4);
    L.cell_first = o; o += align_up(((size_t)n_cells + 2) * 4);        // two-digit partition of compact slots: first slot of every cell
    L.unit_start = o; o += align_up(((size_t)n_cells + 1) * 4);
    L.units = o; o += align_up((size_t)L.max_units * sizeof(Unit));
    L.units_big = o; o += align_up((size_t)L.max_units * sizeof(Unit));
    L.dedup_blocks = (n + kDedupTile - 1) / kDedupTile + 1;
    L.scan_state = o; o += align_up((size_t)L.dedup_blocks * 8);
    L.totals32 = o; o += align_up((size_t)4 * kTotalsMaxPpad * 4);
    L.scalars = o; o += 256;
    L.total = o;
    return true;
}

struct DevBuf { void *p = nullptr; size_t cap = 0; };

struct HostSlot {
    DevBuf in[9], planes, qc, stats, totals, ovf;
    cudaEvent_t in_done = nullptr, compute_done = nullptr, out_done = nullptr;
    mgatk_outputs host = {};          // the caller's buffers of the batch in flight
    uint32_t serial = 0;
    bool busy = false;
};

}  // namespace

struct mgatk_handle {
    int device = 0;
    int sm_count = 148;
    std::string err;
    int64_t launches = 0;
    // stage timing
    cudaEvent_t ev[kMaxStages + 1] = {};
    const char *stage_names[kMaxStages] = {};
    int n_stages = 0;
    bool events_ready = false;
    // host entry points: two slots of device buffers (inputs + outputs) so that the upload of one batch, the kernels
    // of another and the download of a third overlap (mgatk_pileup_host_submit / _wait); the workspace is shared
    // because the kernels of all batches run in order on `stream`
    HostSlot slot[2];
    DevBuf ws;
    uint32_t serial = 0;
    cudaStream_t stream = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    // streaming (mgatk_stream_begin_device .. _finish_device): carry planes for cells with entries beyond 65535
    DevBuf deep_planes, deep_map;
    int deep_cap = 0; int32_t deep_cells = 0; int deep_ppad = 0;
    const void *deep_owner = nullptr;                    // the planes of the stream the carry planes belong to
    // side stream of the overflow-list kernel (runs next to the main pileup kernel): fork / join events
    cudaStream_t side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // variant statistics: hash table of the overflow list of the result being reduced
    DevBuf var_table;
    // clones: x [n][vpad] and inv [n] of the rows being searched
    DevBuf clone_x;
    // clone markers: the nonzero (x, label) pairs of every variant, the fallback's ping-pong pairs, the counters
    DevBuf marker_scratch;
    // deletions: sorted deletions, start bitmap, list of relevant records, dedup table
    DevBuf del_scratch;
};

namespace {

int fail(mgatk_handle *h, int code, const std::string &msg) { if (h) h->err = msg; return code; }

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(h, MGATK_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));    \
    } while (0)

__global__ void k_init(mgatk_stats *stats, int64_t n_records, int32_t *work_counter, u32 *ticket, int accumulate) {
    work_counter[4] = 0; work_counter[5] = 0;            // overflow list: length, work counter (scalars + 32, + 36)
    work_counter[6] = 0;                                 // long-run flag of k_find_long_runs (scalars + 40)
    if (accumulate) stats->total_reads += (uint64_t)n_records;    // streamed batch: the counters keep running
    else {
        stats->total_reads = (uint64_t)n_records;        // readers.py:93 counts every fetched record
        stats->stage1_reads = 0; stats->filtered_reads = 0; stats->dup_with_length = 0;
        stats->dup_position_only = 0; stats->n_empty_seq = 0; stats->n_overflow = 0; stats->error_bits = 0;
    }
    *work_counter = 0;
    *ticket = 0;
}
#if !MGATK_FUSED_SMALL
__global__ void k_publish_m(mgatk_stats *stats, const int64_t *m, int accumulate) {
    stats->stage1_reads = (accumulate ? stats->stage1_reads : 0) + (uint64_t)*m;
}
#endif

void mark(mgatk_handle *h, cudaStream_t s, const char *name) {
    if (h->n_stages < kMaxStages) {
        h->stage_names[h->n_stages] = name;
        cudaEventRecord(h->ev[h->n_stages + 1], s);
        h->n_stages++;
    }
}

// histogram of the pass's digit per chunk and its exclusive scan in (digit, chunk) order
template <class Src>
int histogram_and_scan(mgatk_handle *h, cudaStream_t s, const Src &src, const Layout &L, int pass, char *ws, int64_t *m_out) {
    const int bins = 1 << L.bits[pass];
    u32 *mat = (u32 *)(ws + L.mat), *part = (u32 *)(ws + L.part);
    dim3 sg((bins + 255) / 256, L.ngroups);
#if MGATK_FUSED_SMALL
    u32 *bintot = part + (size_t)L.ngroups * bins;       // [bins + 1]: bin totals, then their exclusive scan (the spare row of `part`)
    k_hist<Src><<<L.nchunks, kHistThreads, (size_t)bins * 4, s>>>(src, L.chunk, L.nchunks, L.shift[pass], bins, mat, bintot);
    k_scan_group_sums<<<sg, 256, 0, s>>>(mat, L.nchunks, bins, part, bintot);
    k_scan_cells<<<1, 1024, 0, s>>>(bintot, bins, m_out);
    k_scan_apply<<<sg, 256, 0, s>>>(mat, L.nchunks, bins, part, bintot);
#else
    k_hist<Src><<<L.nchunks, kHistThreads, (size_t)bins * 4, s>>>(src, L.chunk, L.nchunks, L.shift[pass], bins, mat, nullptr);
    k_scan_group_sums<<<sg, 256, 0, s>>>(mat, L.nchunks, bins, part, nullptr);
    k_scan_bases<<<1, 1024, 0, s>>>(part, L.ngroups, bins, m_out);
    k_scan_apply<<<sg, 256, 0, s>>>(mat, L.nchunks, bins, part, nullptr);
#endif
    h->launches += 4;
    CU(cudaGetLastError());
    return MGATK_OK;
}

// bytes of one per-warp blob staging buffer of the scatter: what 32 blobs of the batch's average size need, with headroom
int warp_buffer_for(const mgatk_batch *b) {
    const int64_t avg = b->n_records > 0 ? (b->blob_bytes / b->n_records + 15) / 16 * 16 : 80;
    int64_t w = 32 * (avg > 16 ? avg : 16) * 5 / 4;
    const int64_t lo = 2560, hi = env_int("MGATK_WBUF_MAX", 10240);
    w = w < lo ? lo : w > hi ? hi : w;
    return (int)((w + 127) / 128 * 128);
}

template <bool kCompact, int kGroups, bool kQualAnd>
int launch_scatter_q(mgatk_handle *h, cudaStream_t s, const ScatterArgs &a) {
    constexpr int kT = kCompact ? kPartThreads : kWideThreads;
    const size_t smem = scatter_smem_bytes<kT>(a.bins, a.wbuf, a.words, kCompact);
    CU(cudaFuncSetAttribute(k_scatter_planes<kCompact, kT, kGroups, kQualAnd>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_scatter_planes<kCompact, kT, kGroups, kQualAnd><<<a.nchunks, kT, smem, s>>>(a);
    h->launches += 1;
    CU(cudaGetLastError());
    return MGATK_OK;
}

template <bool kCompact, int kGroups>
int launch_scatter(mgatk_handle *h, cudaStream_t s, const ScatterArgs &a) {
#if MGATK_LUT_PLANES && MGATK_QUAL_AND
    // min_base_quality in [0, 127] - every real run: the instance whose quality test knows it (two instructions fewer per
    // eight bases); anything else (a negative threshold, one nothing passes) takes the general instance
    if (a.min_baseq >= 0 && a.min_baseq <= 127) return launch_scatter_q<kCompact, kGroups, true>(h, s, a);
#endif
    return launch_scatter_q<kCompact, kGroups, false>(h, s, a);
}

constexpr int kChrMPpad = (int)MGATK_POS_PAD(16569);    // the plane pitch of chrM is compiled in

template <bool kCompact, int kPpad, bool kAcc>
int launch_pileup_t(mgatk_handle *h, cudaStream_t s, const PileupArgs &a, const PileupArgs &a_big, int stage_bytes) {
    const size_t smem_main = (size_t)PileupStages<kCompact>::value * (stage_bytes + range_table_bytes(a.ppad)), smem_big = (size_t)stage_bytes;
    CU(cudaFuncSetAttribute(k_pileup_main<kCompact, kPpad, kAcc>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_main));
    CU(cudaFuncSetAttribute(k_pileup_big<kCompact, kPpad>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_big));
    int per_sm = 0, per_sm_big = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_pileup_main<kCompact, kPpad, kAcc>, kThreads + 32, smem_main));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_big, k_pileup_big<kCompact, kPpad>, kThreads, smem_big));
    if (per_sm < 1) per_sm = 1;
    if (per_sm_big < 1) per_sm_big = 1;
    // The list of big units is usually short or empty: its kernel goes first on a side stream, most of its CTAs leave at
    // once and the CTAs of the main kernel take their place, so both run side by side (they write disjoint tiles).
    if (!h->side) {
        CU(cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    }
    CU(cudaEventRecord(h->ev_fork, s));
    CU(cudaStreamWaitEvent(h->side, h->ev_fork, 0));
    k_pileup_big<kCompact, kPpad><<<h->sm_count * per_sm_big, kThreads, smem_big, h->side>>>(a_big);
    CU(cudaEventRecord(h->ev_join, h->side));
    k_pileup_main<kCompact, kPpad, kAcc><<<h->sm_count * per_sm, kThreads + 32, smem_main, s>>>(a, stage_bytes);   // persistent CTAs pulling units
    CU(cudaStreamWaitEvent(s, h->ev_join, 0));
    h->launches += 2;
    CU(cudaGetLastError());
    return MGATK_OK;
}

template <int kPpad, bool kAcc>
int launch_pileup_p(mgatk_handle *h, cudaStream_t s, bool compact, const PileupArgs &a, const PileupArgs &a_big, int stage_bytes) {
    return compact ? launch_pileup_t<true, kPpad, kAcc>(h, s, a, a_big, stage_bytes) : launch_pileup_t<false, kPpad, kAcc>(h, s, a, a_big, stage_bytes);
}

// the instance of the main kernel: slot layout, chrM's plane pitch or any other, streaming (accumulate) or not
int launch_pileup(mgatk_handle *h, cudaStream_t s, bool compact, const PileupArgs &a, const PileupArgs &a_big, int stage_bytes) {
    if (a.ppad == kChrMPpad)
        return a.accumulate ? launch_pileup_p<kChrMPpad, true>(h, s, compact, a, a_big, stage_bytes)
                            : launch_pileup_p<kChrMPpad, false>(h, s, compact, a, a_big, stage_bytes);
    return a.accumulate ? launch_pileup_p<0, true>(h, s, compact, a, a_big, stage_bytes)
                        : launch_pileup_p<0, false>(h, s, compact, a, a_big, stage_bytes);
}

int validate(mgatk_handle *h, const mgatk_params *p, const mgatk_batch *b, const mgatk_outputs *o) {
    if (!h || !p || !b || !o) return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (b->n_records < 0 || p->n_cells < 0 || p->mito_length <= 0 || b->blob_bytes < 0 || o->overflow_capacity < 0)
        return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (p->dedup_mode < 0 || p->dedup_mode > 2) return fail(h, MGATK_ERR_BAD_ARG, "dedup_mode must be 0, 1 or 2");
    if (p->mito_length >= (1 << 24)) return fail(h, MGATK_ERR_RANGE, "mito_length must be below 2^24");
    if (b->n_records >= (int64_t)0x7fffff00) return fail(h, MGATK_ERR_RANGE, "at most 2^31-257 records per batch");
    if (b->n_records > 0 && (!b->pos || !b->tlen || !b->flag || !b->mapq || !b->bc_idx || !b->l_seq || !b->n_cigar || !b->blob_off))
        return fail(h, MGATK_ERR_BAD_ARG, "null batch array");
    if (b->blob_bytes > 0 && !b->blob) return fail(h, MGATK_ERR_BAD_ARG, "null blob");
    if (((uintptr_t)b->blob & 15) != 0) return fail(h, MGATK_ERR_BAD_ARG, "blob must be 16-byte aligned");
    if (!o->stats || (p->n_cells > 0 && (!o->planes || !o->cell_qc)) || !o->base_totals)
        return fail(h, MGATK_ERR_BAD_ARG, "null output array");
    if (o->overflow_capacity > 0 && !o->overflow) return fail(h, MGATK_ERR_BAD_ARG, "null overflow list");
    if (p->max_read_extent < 1) return fail(h, MGATK_ERR_BAD_ARG, "max_read_extent must be >= 1");
    if (p->max_read_extent > (1 << 20))
        return fail(h, MGATK_ERR_EXTENT, "max_read_extent above 2^20");
    return MGATK_OK;
}

int run_device(mgatk_handle *h, const mgatk_params *p, const mgatk_batch *b, const mgatk_outputs *o, void *ws_v,
               int64_t ws_bytes, cudaStream_t s) {
    int rc = validate(h, p, b, o);
    if (rc) return rc;
    Layout L;
    if (!make_layout(b->n_records, p->n_cells, p->max_read_extent, L)) return fail(h, MGATK_ERR_RANGE, "n_records / n_cells outside limits");
    if ((int64_t)L.total > ws_bytes || !ws_v) return fail(h, MGATK_ERR_WORKSPACE, "workspace too small");
    char *ws = (char *)ws_v;
    CU(cudaSetDevice(h->device));
    if (!h->events_ready) {
        for (int i = 0; i <= kMaxStages; i++) CU(cudaEventCreate(&h->ev[i]));
        h->events_ready = true;
    }
    h->launches = 0; h->n_stages = 0;
    cudaEventRecord(h->ev[0], s);

    const int P = p->mito_length, ppad = (int)MGATK_POS_PAD(P), C = p->n_cells;
    int64_t *m_ptr = (int64_t *)(ws + L.scalars);
    int32_t *n_units = (int32_t *)(ws + L.scalars + 8);
    int32_t *work_counter = (int32_t *)(ws + L.scalars + 16);
    u32 *ticket = (u32 *)(ws + L.scalars + 20);
    int64_t *n_proc = (int64_t *)(ws + L.scalars + 24);
    u64 *error_bits = (u64 *)&o->stats->error_bits;

    const int accumulate = (p->flags & MGATK_FLAG_ACCUMULATE) ? 1 : 0;      // streamed batch: outputs keep accumulating
    k_init<<<1, 1, 0, s>>>(o->stats, b->n_records, work_counter, ticket, accumulate);
    h->launches++;
    if (!accumulate) {
        CU(cudaMemsetAsync(o->base_totals, 0, sizeof(int64_t) * (size_t)P * 4, s));
        if (C > 0) CU(cudaMemsetAsync(o->cell_qc, 0, sizeof(mgatk_cell_qc) * (size_t)C, s));
    } else if (C > 0) {
        k_clear_parked<<<(C + 255) / 256, 256, 0, s>>>(o->cell_qc, C);
        h->launches++;
    }
    if (C == 0) { mark(h, s, "init"); return MGATK_OK; }
    // a cell that is below min_reads_per_cell so far may pass it with a later batch: the gate waits for the finish pass
    const int min_reads = accumulate ? 0 : p->min_reads_per_cell;
    const bool compact = L.fmt.compact != 0;

    // ---- stage 1 + stage 3: filter, reference-coordinate planes, partition by cell ----
    SrcUser su; su.b = *b; su.n_cells = C;
    su.vec4 = (((uintptr_t)b->bc_idx & 15) == 0 && ((uintptr_t)b->flag & 7) == 0) ? 1 : 0;
    uint8_t *slots_a = (uint8_t *)(ws + L.slots[0]), *slots_b = (uint8_t *)(ws + L.slots[1]);
    if ((rc = histogram_and_scan(h, s, su, L, 0, ws, m_ptr))) return rc;
    ScatterArgs sa;
    sa.b = *b; sa.n_cells = C; sa.chunk = L.chunk; sa.nchunks = L.nchunks; sa.shift = L.shift[0]; sa.bins = 1 << L.bits[0];
    sa.mat = (const u32 *)(ws + L.mat); sa.dst = slots_a; sa.error_bits = error_bits;
    sa.words = L.fmt.words; sa.slot_bytes = L.fmt.bytes;
    sa.min_baseq = p->min_baseq; sa.dist = p->min_distance_from_end; sa.min_mapq = p->min_mapq; sa.extent = p->max_read_extent;
    sa.wbuf = warp_buffer_for(b);
    sa.hi_shift = L.passes == 2 ? L.bits[0] : 31;
    {   // the longest window of the batch ends at max_read_extent - min_distance_from_end (pileup.py:67-72)
        const int reach = p->max_read_extent - (p->min_distance_from_end > 0 ? p->min_distance_from_end : 0);
        if (!compact) rc = launch_scatter<false, 7>(h, s, sa);
        else if (reach <= 40) rc = launch_scatter<true, 5>(h, s, sa);
        else if (reach <= 48) rc = launch_scatter<true, 6>(h, s, sa);
        else rc = launch_scatter<true, 7>(h, s, sa);
        if (rc) return rc;
    }
    uint8_t *grouped = slots_a, *piled = slots_b;
    if (L.passes == 2) {
        SrcSlots ss; ss.a = slots_a; ss.m = m_ptr; ss.slot_bytes = L.fmt.bytes; ss.compact = compact; ss.hi_shift = L.bits[0];
        if ((rc = histogram_and_scan(h, s, ss, L, 1, ws, nullptr))) return rc;
        const int bins = 1 << L.bits[1];
        k_scatter_slots<<<L.nchunks, kPartThreads, rank_smem_bytes(bins), s>>>(ss, L.chunk, L.nchunks, L.shift[1], bins, (const u32 *)(ws + L.mat), slots_b);
        h->launches += 1;
        CU(cudaGetLastError());
        grouped = slots_b; piled = slots_a;
    }
#if !MGATK_FUSED_SMALL
    k_publish_m<<<1, 1, 0, s>>>(o->stats, m_ptr, accumulate);
    h->launches += 1;
#endif
    mark(h, s, "filter+planes+partition");

    // ---- stage 2: dedup, mapq gate, compaction of the reads to pile up ----
    int32_t *cell_start = (int32_t *)(ws + L.cell_start);
    CU(cudaMemsetAsync(ws + L.scan_state, 0, (size_t)L.dedup_blocks * 8, s));
    DedupArgs da;
    da.slots = grouped; da.out = piled; da.slot_bytes = L.fmt.bytes; da.m_ptr = m_ptr;
    da.cell_first = (const u32 *)(ws + L.mat); da.n_first = 1 << L.bits[0];      // row 0 of the scanned histogram (one pass)
    if (compact && L.passes == 2) {                      // no such row after two digit passes: count the slots per cell
        u32 *cf = (u32 *)(ws + L.cell_first);
        CU(cudaMemsetAsync(cf, 0, ((size_t)C + 1) * 4, s));
        const int smem_cells = C < 12288 ? C : 12288;
        k_cell_counts<<<h->sm_count * 2, 1024, (size_t)smem_cells * 4, s>>>(su, smem_cells, cf);
        k_scan_cells<<<1, 1024, 0, s>>>(cf, C);
        h->launches += 2;
        da.cell_first = cf; da.n_first = C;
    }
    da.dedup_mode = p->dedup_mode; da.qc = o->cell_qc; da.stats = o->stats;
    da.ticket = ticket; da.scan_state = (u64 *)(ws + L.scan_state); da.n_proc_out = n_proc;
    {   // very long (cell, start) runs switch k_dedup to its warp-cooperative look-back (scalars + 40: the flag)
        u32 *flag = (u32 *)(ws + L.scalars + 40);
        da.long_runs = flag;
        const unsigned blocks = (unsigned)((b->n_records / kLongRun + 255) / 256 + 1);
        mgatk_stats *pub = MGATK_FUSED_SMALL ? o->stats : nullptr;     // stats.stage1_reads is published by this kernel's first thread
        if (compact) k_find_long_runs<true><<<blocks, 256, 0, s>>>(grouped, L.fmt.bytes, m_ptr, da.cell_first, da.n_first, flag, pub, accumulate);
        else k_find_long_runs<false><<<blocks, 256, 0, s>>>(grouped, L.fmt.bytes, m_ptr, da.cell_first, da.n_first, flag, pub, accumulate);
        h->launches += 1;
    }
    // (developer knob: unused dynamic shared memory caps the resident CTAs per SM - 45 KB: five, 56 KB: four)
    const int dpad = env_int("MGATK_DEDUP_PAD", 0);
    if (dpad > 0) {
        CU(cudaFuncSetAttribute(k_dedup<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dpad));
        CU(cudaFuncSetAttribute(k_dedup<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, dpad));
    }
    if (compact) {
        k_dedup<true, false><<<(unsigned)L.dedup_blocks, kDedupThreads, dpad, s>>>(da);
        k_dedup<true, true><<<(unsigned)L.dedup_blocks, kDedupThreads, 0, s>>>(da);
    } else {
        k_dedup<false, false><<<(unsigned)L.dedup_blocks, kDedupThreads, dpad, s>>>(da);
        k_dedup<false, true><<<(unsigned)L.dedup_blocks, kDedupThreads, 0, s>>>(da);
    }
    h->launches += 2;
    mark(h, s, "dedup");

    // ---- units ----
    int32_t *unit_start = (int32_t *)(ws + L.unit_start);
    Unit *units = (Unit *)(ws + L.units);
    k_plan_scan<<<1, 1024, 0, s>>>(o->cell_qc, C, min_reads, L.unit_reads, ppad, cell_start, unit_start, n_units);
    const SlotList sl{piled, L.fmt.bytes};
    k_plan_units<<<(unsigned)((L.max_units + 255) / 256), 256, 0, s>>>(cell_start, o->cell_qc, sl, unit_start, C,
                                                                      min_reads, L.unit_reads, ppad, p->max_read_extent, units,
                                                                      L.cap_reads, (Unit *)(ws + L.units_big), work_counter + 4);
    h->launches += 2;
    mark(h, s, "plan");

    // ---- stages 4-6 ----
    PileupArgs a;
    a.slots = piled; a.blob = b->blob; a.blob_bytes = b->blob_bytes;
    a.units = units; a.n_units = n_units; a.work_counter = work_counter;
    a.planes = o->planes; a.qc = o->cell_qc; a.stats = o->stats; a.ovf = o->overflow; a.ovf_cap = o->overflow_capacity;
    a.P = P; a.ppad = ppad; a.min_baseq = p->min_baseq; a.dist = p->min_distance_from_end;
    a.max_bias = p->max_strand_bias;
    a.raw = (p->flags & MGATK_FLAG_RAW_PILEUP) ? 1 : 0;
    a.apply_bias = !a.raw && !(p->max_strand_bias >= 1.0);   // max(f,r)/total never exceeds 1.0
    a.accumulate = accumulate;
    a.extent = p->max_read_extent;
    a.slot_bytes = L.fmt.bytes; a.words = L.fmt.words;
    a.cap_reads = L.cap_reads;
    a.deep_map = nullptr; a.deep_planes = nullptr; a.deep_count = nullptr; a.deep_cap = 0;
    if (accumulate && h->deep_owner == (const void *)o->planes && h->deep_cells == C && h->deep_ppad == ppad) {
        a.deep_map = (int32_t *)h->deep_map.p + 1; a.deep_count = (int32_t *)h->deep_map.p;
        a.deep_planes = (u32 *)h->deep_planes.p; a.deep_cap = h->deep_cap;
    }
    // cross-cell base totals: reduced by the counting kernels themselves (32-bit atomics on a [4][ppad] scratch, widened
    // below) when the contig fits the scratch, else by a pass over the finished planes
    const bool fused_totals = !accumulate && ppad <= kTotalsMaxPpad && env_int("MGATK_FUSED_TOTALS", 1);
    a.totals32 = fused_totals ? (u32 *)(ws + L.totals32) : nullptr;
    if (fused_totals) CU(cudaMemsetAsync(a.totals32, 0, (size_t)4 * ppad * 4, s));
    PileupArgs a2 = a;
    a2.units = (Unit *)(ws + L.units_big); a2.n_units = work_counter + 4; a2.work_counter = work_counter + 5;
    rc = launch_pileup(h, s, compact, a, a2, L.stage_bytes);
    if (rc) return rc;
    mark(h, s, "pileup");
    if (accumulate) return MGATK_OK;                     // filters, coverage, statistics: mgatk_stream_finish_device

    // ---- reference-allele totals, median depth ----
    const bool widen_in_median = MGATK_FUSED_SMALL && fused_totals;      // k_median's CTAs widen the totals on their way in
    if (fused_totals) {
        if (!widen_in_median) {
            k_totals_widen<<<(P + 255) / 256, 256, 0, s>>>(a.totals32, P, ppad, (u64 *)o->base_totals);
            h->launches++;
        }
    } else {
        dim3 tg((ppad / 2 + 127) / 128, min((C + kTotalsCellGroup - 1) / kTotalsCellGroup, 65535));
        k_base_totals<<<tg, 128, 0, s>>>(o->planes, C, P, ppad, (u64 *)o->base_totals);
        h->launches++;
        if (o->overflow_capacity > 0) {
            k_base_totals_overflow<<<8, 256, 0, s>>>(o->overflow, o->stats, o->overflow_capacity, P, (u64 *)o->base_totals);
            h->launches++;
        }
    }
    k_median<<<C, 256, 0, s>>>(o->planes, P, ppad, o->cell_qc, o->overflow_capacity > 0 ? o->overflow : nullptr, o->stats, o->overflow_capacity,
                               widen_in_median ? a.totals32 : nullptr, (u64 *)o->base_totals);
    h->launches++;
    CU(cudaGetLastError());
    mark(h, s, "totals+median");
    return MGATK_OK;
}

int ensure(mgatk_handle *h, DevBuf &b, size_t bytes) {
    if (bytes <= b.cap && b.p) return MGATK_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
    size_t want = bytes < 256 ? 256 : bytes;
    CU(cudaMalloc(&b.p, want));
    b.cap = want;
    return MGATK_OK;
}

template <class T>
int filter_planes(mgatk_handle *h, T *planes_dev, int32_t n_cells, int32_t mito_length, double max_strand_bias, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!planes_dev || n_cells < 0 || mito_length <= 0) return fail(h, MGATK_ERR_BAD_ARG, "bad argument");
    if (n_cells == 0) return MGATK_OK;
    CU(cudaSetDevice(h->device));
    dim3 grid((mito_length + 255) / 256, n_cells < 65535 ? n_cells : 65535);
    k_filter_planes<T><<<grid, 256, 0, (cudaStream_t)stream>>>(planes_dev, n_cells, mito_length, (int)MGATK_POS_PAD(mito_length), max_strand_bias);
    h->launches = 1;
    CU(cudaGetLastError());
    return MGATK_OK;
}

// checks shared by the variant entries; builds the overflow lookup table of `o` on `s` (*table: nullptr without a list)
int variant_prepare(mgatk_handle *h, const mgatk_params *p, const mgatk_outputs *o, cudaStream_t s, const OvfSlot **table) {
    *table = nullptr;
    if (!p || !o) return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (p->n_cells < 0 || p->mito_length <= 0 || o->overflow_capacity < 0) return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (p->mito_length >= (1 << 24)) return fail(h, MGATK_ERR_RANGE, "mito_length must be below 2^24");
    if (!o->stats || !o->base_totals || (p->n_cells > 0 && !o->planes)) return fail(h, MGATK_ERR_BAD_ARG, "null result array");
    if (o->overflow_capacity > 0 && !o->overflow) return fail(h, MGATK_ERR_BAD_ARG, "null overflow list");
    if (o->overflow_capacity > (int64_t)1 << 30) return fail(h, MGATK_ERR_RANGE, "overflow_capacity above 2^30");
    CU(cudaSetDevice(h->device));
    if (o->overflow_capacity == 0 || p->n_cells == 0) return MGATK_OK;
    const u64 slots = ovf_table_slots((u64)o->overflow_capacity);
    int rc = ensure(h, h->var_table, (size_t)slots * sizeof(OvfSlot));
    if (rc) return rc;
    OvfSlot *t = (OvfSlot *)h->var_table.p;
    const unsigned clear_blocks = (unsigned)((slots + 255) / 256 < 1024 ? (slots + 255) / 256 : 1024);
    const unsigned insert_blocks = (unsigned)((o->overflow_capacity + 255) / 256 < 1024 ? (o->overflow_capacity + 255) / 256 : 1024);
    k_ovf_clear<<<clear_blocks, 256, 0, s>>>(t, o->stats, o->overflow_capacity);
    k_ovf_insert<<<insert_blocks, 256, 0, s>>>(t, o->overflow, o->stats, o->overflow_capacity);
    CU(cudaGetLastError());
    *table = t;
    return MGATK_OK;
}

}  // namespace

extern "C" {

int mgatk_abi_version(void) { return MGATK_ABI_VERSION; }

const char *mgatk_status_string(int status) {
    switch (status) {
        case MGATK_OK: return "ok";
        case MGATK_ERR_BAD_ARG: return "bad argument";
        case MGATK_ERR_CUDA: return "CUDA error";
        case MGATK_ERR_WORKSPACE: return "workspace too small";
        case MGATK_ERR_UNSORTED: return "records are not sorted by reference_start";
        case MGATK_ERR_EXTENT: return "a read exceeds max_read_extent";
        case MGATK_ERR_OVERFLOW_CAP: return "overflow list capacity exceeded";
        case MGATK_ERR_NO_DEVICE: return "no usable CUDA device";
        case MGATK_ERR_RANGE: return "size outside supported range";
        case MGATK_ERR_STREAM_SATURATED: return "streaming: more cells with entries beyond 65535 than carry-plane sets";
        default: return "unknown status";
    }
}

int mgatk_create(mgatk_handle **out, int device) {
    if (!out) return MGATK_ERR_BAD_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return MGATK_ERR_NO_DEVICE;
    mgatk_handle *h = new mgatk_handle();
    h->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete h; return MGATK_ERR_NO_DEVICE; }
    h->sm_count = prop.multiProcessorCount;
    *out = h;
    return MGATK_OK;
}

int mgatk_destroy(mgatk_handle *h) {
    if (!h) return MGATK_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (HostSlot &sl : h->slot) {
        DevBuf *all[] = {&sl.planes, &sl.qc, &sl.stats, &sl.totals, &sl.ovf};
        for (DevBuf *b : all) if (b->p) cudaFree(b->p);
        for (DevBuf &b : sl.in) if (b.p) cudaFree(b.p);
        if (sl.in_done) { cudaEventDestroy(sl.in_done); cudaEventDestroy(sl.compute_done); cudaEventDestroy(sl.out_done); }
    }
    if (h->ws.p) cudaFree(h->ws.p);
    if (h->deep_planes.p) cudaFree(h->deep_planes.p);
    if (h->deep_map.p) cudaFree(h->deep_map.p);
    if (h->var_table.p) cudaFree(h->var_table.p);
    if (h->clone_x.p) cudaFree(h->clone_x.p);
    if (h->marker_scratch.p) cudaFree(h->marker_scratch.p);
    if (h->del_scratch.p) cudaFree(h->del_scratch.p);
    if (h->s_h2d) { cudaStreamDestroy(h->s_h2d); cudaStreamDestroy(h->s_d2h); }
    if (h->events_ready) for (int i = 0; i <= kMaxStages; i++) cudaEventDestroy(h->ev[i]);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->side) { cudaStreamDestroy(h->side); cudaEventDestroy(h->ev_fork); cudaEventDestroy(h->ev_join); }
    delete h;
    return MGATK_OK;
}

const char *mgatk_last_error(const mgatk_handle *h) { return h ? h->err.c_str() : "null handle"; }

int64_t mgatk_workspace_bytes(int64_t n_records, int32_t n_cells, int32_t max_read_extent) {
    Layout L;
    if (!make_layout(n_records, n_cells, max_read_extent, L)) return -1;
    return (int64_t)L.total;
}

int mgatk_pileup_device(mgatk_handle *h, const mgatk_params *params, const mgatk_batch *batch_dev,
                        const mgatk_outputs *out_dev, void *workspace_dev, int64_t workspace_bytes, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    return run_device(h, params, batch_dev, out_dev, workspace_dev, workspace_bytes, (cudaStream_t)stream);
}

int mgatk_filter_strand_bias_device(mgatk_handle *h, uint16_t *planes_dev, int32_t n_cells, int32_t mito_length,
                                    double max_strand_bias, void *stream) {
    return filter_planes<uint16_t>(h, planes_dev, n_cells, mito_length, max_strand_bias, stream);
}

int mgatk_filter_strand_bias_u32_device(mgatk_handle *h, uint32_t *planes_dev, int32_t n_cells, int32_t mito_length,
                                        double max_strand_bias, void *stream) {
    return filter_planes<uint32_t>(h, planes_dev, n_cells, mito_length, max_strand_bias, stream);
}

int mgatk_stream_begin_device(mgatk_handle *h, const mgatk_params *p, const mgatk_outputs *o, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!p || !o || !o->stats || !o->base_totals || p->n_cells < 0 || p->mito_length <= 0 || (p->n_cells > 0 && (!o->planes || !o->cell_qc)))
        return fail(h, MGATK_ERR_BAD_ARG, "bad argument");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t C = (size_t)p->n_cells, P = (size_t)p->mito_length, ppad = (size_t)MGATK_POS_PAD(P);
    if (C) CU(cudaMemsetAsync(o->planes, 0, C * MGATK_N_PLANES * ppad * 2, s));
    if (C) CU(cudaMemsetAsync(o->cell_qc, 0, C * sizeof(mgatk_cell_qc), s));
    if (C) {    // carry planes for up to kDeepSets cells whose entries pass 65535 while the batches add up (bulk mode, deep piles)
        int rc;
        const int cap = (int)(C < (size_t)env_int("MGATK_DEEP_SETS", 64) ? C : (size_t)env_int("MGATK_DEEP_SETS", 64));
        if ((rc = ensure(h, h->deep_map, (C + 1) * 4)) || (rc = ensure(h, h->deep_planes, (size_t)cap * 10 * ppad * 4))) return rc;
        CU(cudaMemsetAsync(h->deep_map.p, 0xff, (C + 1) * 4, s));
        CU(cudaMemsetAsync(h->deep_map.p, 0, 4, s));                             // word 0: sets handed out
        CU(cudaMemsetAsync(h->deep_planes.p, 0, (size_t)cap * 10 * ppad * 4, s));
        h->deep_cap = cap; h->deep_cells = (int32_t)C; h->deep_ppad = (int)ppad; h->deep_owner = o->planes;
    }
    CU(cudaMemsetAsync(o->stats, 0, sizeof(mgatk_stats), s));
    CU(cudaMemsetAsync(o->base_totals, 0, P * 4 * sizeof(int64_t), s));
    return MGATK_OK;
}

int mgatk_stream_finish_device(mgatk_handle *h, const mgatk_params *p, const mgatk_outputs *o, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!p || !o || !o->stats || !o->base_totals || p->n_cells < 0 || p->mito_length <= 0 || (p->n_cells > 0 && (!o->planes || !o->cell_qc)))
        return fail(h, MGATK_ERR_BAD_ARG, "bad argument");
    if (o->overflow_capacity > 0 && !o->overflow) return fail(h, MGATK_ERR_BAD_ARG, "null overflow list");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int C = p->n_cells, P = p->mito_length, ppad = (int)MGATK_POS_PAD(P);
    h->launches = 0;
    if (C == 0) return MGATK_OK;
    PileupArgs a;
    memset(&a, 0, sizeof(a));
    a.planes = o->planes; a.qc = o->cell_qc; a.stats = o->stats; a.ovf = o->overflow; a.ovf_cap = o->overflow_capacity;
    a.P = P; a.ppad = ppad; a.max_bias = p->max_strand_bias;
    a.raw = (p->flags & MGATK_FLAG_RAW_PILEUP) ? 1 : 0;
    a.apply_bias = !a.raw && !(p->max_strand_bias >= 1.0);
    if (h->deep_owner == (const void *)o->planes && h->deep_cells == C && h->deep_ppad == ppad) {
        a.deep_map = (int32_t *)h->deep_map.p + 1; a.deep_count = (int32_t *)h->deep_map.p;
        a.deep_planes = (u32 *)h->deep_planes.p; a.deep_cap = h->deep_cap;
    }
    k_clear_parked<<<(C + 255) / 256, 256, 0, s>>>(o->cell_qc, C);
    k_stream_finish<<<h->sm_count * 8, 256, 0, s>>>(a, C, p->min_reads_per_cell);
    dim3 tg((ppad / 2 + 127) / 128, min((C + kTotalsCellGroup - 1) / kTotalsCellGroup, 65535));
    k_base_totals<<<tg, 128, 0, s>>>(o->planes, C, P, ppad, (u64 *)o->base_totals);
    h->launches += 3;
    if (o->overflow_capacity > 0) {
        k_base_totals_overflow<<<8, 256, 0, s>>>(o->overflow, o->stats, o->overflow_capacity, P, (u64 *)o->base_totals);
        h->launches++;
    }
    k_median<<<C, 256, 0, s>>>(o->planes, P, ppad, o->cell_qc, o->overflow_capacity > 0 ? o->overflow : nullptr, o->stats, o->overflow_capacity,
                               nullptr, nullptr);
    h->launches++;
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_check_stats(const mgatk_stats *st) {
    if (!st) return MGATK_ERR_BAD_ARG;
    if (st->error_bits & ERR_UNSORTED) return MGATK_ERR_UNSORTED;
    if (st->error_bits & ERR_EXTENT) return MGATK_ERR_EXTENT;
    if (st->error_bits & ERR_OVERFLOW_CAP) return MGATK_ERR_OVERFLOW_CAP;
    if (st->error_bits & ERR_SATURATED) return MGATK_ERR_STREAM_SATURATED;
    if (st->error_bits & ERR_DEL_RANGE) return MGATK_ERR_RANGE;
    return MGATK_OK;
}

int mgatk_pileup_host_submit(mgatk_handle *h, const mgatk_params *p, const mgatk_batch *b, const mgatk_outputs *o,
                             int64_t *ticket) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!ticket) return fail(h, MGATK_ERR_BAD_ARG, "null ticket");
    *ticket = -1;
    int rc = validate(h, p, b, o);
    if (rc) return rc;
    const int k_slot = !h->slot[0].busy ? 0 : !h->slot[1].busy ? 1 : -1;
    if (k_slot < 0) return fail(h, MGATK_ERR_BAD_ARG, "two batches in flight: wait for the older ticket first");
    HostSlot &sl = h->slot[k_slot];
    CU(cudaSetDevice(h->device));
    if (!h->stream) CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    if (!h->s_h2d) {
        CU(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    }
    if (!sl.in_done) {
        CU(cudaEventCreateWithFlags(&sl.in_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&sl.compute_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&sl.out_done, cudaEventDisableTiming));
    }
    const size_t n = (size_t)b->n_records, C = (size_t)p->n_cells, P = (size_t)p->mito_length;
    const size_t ppad = (size_t)MGATK_POS_PAD(P);
    const size_t planes_bytes = C * MGATK_N_PLANES * ppad * 2;
    const int64_t ws_bytes = mgatk_workspace_bytes(b->n_records, p->n_cells, p->max_read_extent);
    if (ws_bytes < 0) return fail(h, MGATK_ERR_RANGE, "n_records / n_cells outside limits");
    const void *src[9] = {b->pos, b->tlen, b->flag, b->mapq, b->bc_idx, b->l_seq, b->n_cigar, b->blob_off, b->blob};
    const size_t bytes[9] = {4 * n, 4 * n, 2 * n, n, 4 * n, 2 * n, 2 * n, 4 * n, (size_t)b->blob_bytes};
    // (a growing buffer is freed and reallocated: cudaFree waits for the device, so nothing in flight loses its memory;
    //  the workspace grows only while no other batch is in flight)
    if ((size_t)ws_bytes > h->ws.cap && h->slot[k_slot ^ 1].busy) CU(cudaEventSynchronize(h->slot[k_slot ^ 1].compute_done));
    for (int k = 0; k < 9; k++)
        if ((rc = ensure(h, sl.in[k], bytes[k]))) return rc;
    if ((rc = ensure(h, sl.planes, planes_bytes)) || (rc = ensure(h, sl.qc, C * sizeof(mgatk_cell_qc))) ||
        (rc = ensure(h, sl.stats, sizeof(mgatk_stats))) || (rc = ensure(h, sl.totals, P * 4 * 8)) ||
        (rc = ensure(h, sl.ovf, (size_t)o->overflow_capacity * sizeof(mgatk_overflow))) ||
        (rc = ensure(h, h->ws, (size_t)ws_bytes)))
        return rc;
    // upload
    for (int k = 0; k < 9; k++)
        if (bytes[k]) CU(cudaMemcpyAsync(sl.in[k].p, src[k], bytes[k], cudaMemcpyHostToDevice, h->s_h2d));
    CU(cudaEventRecord(sl.in_done, h->s_h2d));
    // kernels
    cudaStream_t s = h->stream;
    CU(cudaStreamWaitEvent(s, sl.in_done, 0));
    mgatk_batch bd = *b;
    bd.pos = (const int32_t *)sl.in[0].p; bd.tlen = (const int32_t *)sl.in[1].p; bd.flag = (const uint16_t *)sl.in[2].p;
    bd.mapq = (const uint8_t *)sl.in[3].p; bd.bc_idx = (const int32_t *)sl.in[4].p; bd.l_seq = (const uint16_t *)sl.in[5].p;
    bd.n_cigar = (const uint16_t *)sl.in[6].p; bd.blob_off = (const uint32_t *)sl.in[7].p; bd.blob = (const uint8_t *)sl.in[8].p;
    mgatk_outputs od = *o;
    od.planes = (uint16_t *)sl.planes.p; od.cell_qc = (mgatk_cell_qc *)sl.qc.p; od.stats = (mgatk_stats *)sl.stats.p;
    od.base_totals = (int64_t *)sl.totals.p; od.overflow = o->overflow_capacity ? (mgatk_overflow *)sl.ovf.p : nullptr;
    rc = run_device(h, p, &bd, &od, h->ws.p, ws_bytes, s);
    if (rc) { cudaStreamSynchronize(h->s_h2d); cudaStreamSynchronize(s); return rc; }   // nothing of this batch stays in flight
    CU(cudaEventRecord(sl.compute_done, s));
    // download
    CU(cudaStreamWaitEvent(h->s_d2h, sl.compute_done, 0));
    if (planes_bytes) CU(cudaMemcpyAsync(o->planes, od.planes, planes_bytes, cudaMemcpyDeviceToHost, h->s_d2h));
    if (C) CU(cudaMemcpyAsync(o->cell_qc, od.cell_qc, C * sizeof(mgatk_cell_qc), cudaMemcpyDeviceToHost, h->s_d2h));
    CU(cudaMemcpyAsync(o->stats, od.stats, sizeof(mgatk_stats), cudaMemcpyDeviceToHost, h->s_d2h));
    CU(cudaMemcpyAsync(o->base_totals, od.base_totals, P * 4 * 8, cudaMemcpyDeviceToHost, h->s_d2h));
    CU(cudaEventRecord(sl.out_done, h->s_d2h));
    sl.host = *o; sl.busy = true; sl.serial = ++h->serial;
    *ticket = ((int64_t)sl.serial << 1) | k_slot;
    return MGATK_OK;
}

int mgatk_pileup_host_wait(mgatk_handle *h, int64_t ticket) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (ticket < 0) return fail(h, MGATK_ERR_BAD_ARG, "bad ticket");
    HostSlot &sl = h->slot[ticket & 1];
    if (!sl.busy || (int64_t)sl.serial != (ticket >> 1)) return fail(h, MGATK_ERR_BAD_ARG, "ticket is not in flight");
    CU(cudaSetDevice(h->device));
    sl.busy = false;
    CU(cudaEventSynchronize(sl.out_done));
    const mgatk_outputs *o = &sl.host;
    if (o->overflow_capacity && o->stats->n_overflow) {
        size_t k = (size_t)(o->stats->n_overflow < (uint64_t)o->overflow_capacity ? o->stats->n_overflow : (uint64_t)o->overflow_capacity);
        CU(cudaMemcpyAsync(o->overflow, sl.ovf.p, k * sizeof(mgatk_overflow), cudaMemcpyDeviceToHost, h->s_d2h));
        CU(cudaStreamSynchronize(h->s_d2h));
    }
    int rc = mgatk_check_stats(o->stats);
    if (rc) return fail(h, rc, mgatk_status_string(rc));
    return MGATK_OK;
}

int mgatk_pileup_host(mgatk_handle *h, const mgatk_params *p, const mgatk_batch *b, const mgatk_outputs *o) {
    int64_t ticket = -1;
    int rc = mgatk_pileup_host_submit(h, p, b, o, &ticket);
    if (rc) return rc;
    return mgatk_pileup_host_wait(h, ticket);
}

int mgatk_variant_stats_device(mgatk_handle *h, const mgatk_params *p, const mgatk_outputs *o, const uint8_t *cell_mask_dev,
                               int32_t low_coverage_threshold, mgatk_variant_sums *out_dev, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!out_dev) return fail(h, MGATK_ERR_BAD_ARG, "null output array");
    if (low_coverage_threshold < 1) return fail(h, MGATK_ERR_BAD_ARG, "low_coverage_threshold must be >= 1");
    cudaStream_t s = (cudaStream_t)stream;
    const OvfSlot *table = nullptr;
    int rc = variant_prepare(h, p, o, s, &table);
    if (rc) return rc;
    VarArgs a;
    a.planes = o->planes; a.stats = o->stats; a.totals = o->base_totals; a.table = table; a.ovf_cap = o->overflow_capacity;
    a.mask = cell_mask_dev; a.C = p->n_cells; a.P = p->mito_length; a.ppad = (int)MGATK_POS_PAD(p->mito_length);
    a.low = (u32)low_coverage_threshold; a.out = out_dev;
    k_variant_stats<<<(unsigned)((a.P + kVarTile - 1) / kVarTile), kVarWarps * 32, 0, s>>>(a);
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_variant_cells_device(mgatk_handle *h, const mgatk_params *p, const mgatk_outputs *o, const int32_t *variants_dev,
                               int32_t n_variants, uint32_t *out_dev, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (n_variants < 0) return fail(h, MGATK_ERR_BAD_ARG, "negative n_variants");
    if (n_variants > 0 && (!variants_dev || !out_dev)) return fail(h, MGATK_ERR_BAD_ARG, "null variant or output array");
    cudaStream_t s = (cudaStream_t)stream;
    const OvfSlot *table = nullptr;
    int rc = variant_prepare(h, p, o, s, &table);
    if (rc) return rc;
    if (n_variants == 0 || p->n_cells == 0) return MGATK_OK;
    dim3 grid((unsigned)((p->n_cells + 255) / 256), (unsigned)(n_variants < 65535 ? n_variants : 65535));
    k_variant_cells<<<grid, 256, 0, s>>>(o->planes, table, o->stats, o->overflow_capacity, variants_dev, n_variants, p->n_cells,
                                         p->mito_length, (int)MGATK_POS_PAD(p->mito_length), out_dev);
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_clone_knn_device(mgatk_handle *h, const uint32_t *counts_dev, const int32_t *rows_dev, int32_t n_rows,
                           int32_t n_cells, int32_t n_variants, int32_t k, int32_t *nbr_out, double *sim_out, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (k < 2 || k > MGATK_CLONE_K_MAX) return fail(h, MGATK_ERR_BAD_ARG, "k must be in [2, 64]");
    if (n_rows < 0 || n_cells < 0 || n_variants < 0) return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (n_rows == 0) return MGATK_OK;
    if (!rows_dev || !nbr_out || !sim_out || !counts_dev) return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (n_variants == 0 || n_rows > n_cells) return fail(h, MGATK_ERR_BAD_ARG, "graph rows need a variant and distinct cells");
    if (n_rows > MGATK_CLONE_MAX_ROWS || n_variants > MGATK_CLONE_MAX_VARIANTS)
        return fail(h, MGATK_ERR_RANGE, "n_rows above 2^24 or n_variants above 4096");
    const int vpad = clone_vpad(n_variants);
    if ((int64_t)n_rows * vpad > MGATK_CLONE_MAX_ELEMENTS) return fail(h, MGATK_ERR_RANGE, "n_rows * padded n_variants above 2^31");
    CU(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int k_eff = k < n_rows ? k : n_rows;
    if (k_eff == 1) {
        k_clone_self<<<1, 32, 0, s>>>(n_rows, k_eff, nbr_out, sim_out);
        CU(cudaGetLastError());
        return MGATK_OK;
    }
    int rc = ensure(h, h->clone_x, ((size_t)n_rows * vpad + n_rows) * sizeof(double));
    if (rc) return rc;
    double *x = (double *)h->clone_x.p, *inv = x + (size_t)n_rows * vpad;
    k_clone_af<<<(unsigned)((n_rows + 127) / 128), 128, 0, s>>>(counts_dev, rows_dev, n_rows, n_cells, n_variants, vpad, x, inv);
    CU(cudaGetLastError());
    const int smem = (int)sizeof(CloneKnnSmem);
    CU(cudaFuncSetAttribute(k_clone_knn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_clone_knn<<<(unsigned)((n_rows + kCloneTile - 1) / kCloneTile), kCloneThreads, smem, s>>>(x, inv, n_rows, vpad, k_eff,
                                                                                                nbr_out, sim_out);
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_clone_snn_device(mgatk_handle *h, const int32_t *nbr_dev, int32_t n, int32_t k_eff, double *w_out, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (n < 0) return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (n == 0) return MGATK_OK;
    if (k_eff < 1 || k_eff > MGATK_CLONE_K_MAX || k_eff > n) return fail(h, MGATK_ERR_BAD_ARG, "k_eff must be in [1, min(64, n)]");
    if (!nbr_dev || !w_out) return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (n > MGATK_CLONE_MAX_ROWS) return fail(h, MGATK_ERR_RANGE, "n above 2^24");
    CU(cudaSetDevice(h->device));
    k_clone_snn<<<(unsigned)((n + kSnnWarps - 1) / kSnnWarps), kSnnWarps * 32, 0, (cudaStream_t)stream>>>(nbr_dev, n, k_eff, w_out);
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_marker_ranks_device(mgatk_handle *h, const uint32_t *counts_dev, const int32_t *labels_dev, int32_t n_cells,
                              int32_t n_variants, int32_t n_groups, uint64_t *rank2_out, uint64_t *ties_out, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (n_cells < 0 || n_variants < 0) return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (n_groups < 1) return fail(h, MGATK_ERR_BAD_ARG, "n_groups must be >= 1");
    if ((n_cells > 0 && !labels_dev) || (n_cells > 0 && n_variants > 0 && !counts_dev) ||
        (n_variants > 0 && (!rank2_out || !ties_out)))
        return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (n_cells > MGATK_MARKER_MAX_CELLS || n_variants > MGATK_CLONE_MAX_VARIANTS)
        return fail(h, MGATK_ERR_RANGE, "n_cells above 2^21 or n_variants above 4096");
    if (n_cells > 0 && n_groups > n_cells) return fail(h, MGATK_ERR_RANGE, "n_groups above n_cells");
    if (n_variants == 0) return MGATK_OK;
    CU(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const size_t V = (size_t)n_variants, C = (size_t)n_cells, G = (size_t)n_groups;
    if (n_cells == 0) {
        CU(cudaMemsetAsync(rank2_out, 0, V * G * sizeof(uint64_t), s));
        CU(cudaMemsetAsync(ties_out, 0, V * sizeof(uint64_t), s));
        return MGATK_OK;
    }
    const int grid = n_variants < 2 * h->sm_count ? n_variants : 2 * h->sm_count;
    const size_t tmp = n_cells > kMarkerS ? (size_t)grid * C : 0;       // the fallback needs ping-pong pairs
    const size_t o_tkeys = align_up(V * C * 8), o_labs = o_tkeys + align_up(tmp * 8), o_tlabs = o_labs + align_up(V * C * 4);
    const size_t o_cnt = o_tlabs + align_up(tmp * 4), n_cnt = V + G + 2;
    int rc = ensure(h, h->marker_scratch, o_cnt + n_cnt * 4);
    if (rc) return rc;
    char *base = (char *)h->marker_scratch.p;
    u32 *nnz = (u32 *)(base + o_cnt), *gsize = nnz + V, *npop = gsize + G + 1;
    CU(cudaMemsetAsync(nnz, 0, n_cnt * 4, s));
    dim3 sg((unsigned)((C + kMarkerSplitThreads - 1) / kMarkerSplitThreads), (unsigned)V);
    k_marker_split<<<sg, kMarkerSplitThreads, 0, s>>>(counts_dev, labels_dev, n_cells, n_groups, nnz, gsize, npop,
                                                      (u64 *)base, (int32_t *)(base + o_labs));
    CU(cudaGetLastError());
    const int smem = (int)sizeof(MarkerSmem);
    CU(cudaFuncSetAttribute(k_marker_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_marker_rank<<<grid, kMarkerThreads, smem, s>>>((u64 *)base, (int32_t *)(base + o_labs), nnz, gsize, npop, n_cells,
                                                     n_variants, n_groups, (u64 *)(base + o_tkeys),
                                                     (int32_t *)(base + o_tlabs), (u64 *)rank2_out, (u64 *)ties_out);
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_deletion_scan_device(mgatk_handle *h, const mgatk_params *p, const mgatk_batch *b, int32_t min_clip,
                               const int32_t *left_dev, const int32_t *right_dev, int32_t n_deletions,
                               uint32_t *counts_out, uint64_t *clip_hist_out, uint64_t *clip_seq_out,
                               uint64_t *error_bits_out, void *stream) {
    if (!h) return MGATK_ERR_BAD_ARG;
    h->err.clear();
    if (!p || !b || !error_bits_out) return fail(h, MGATK_ERR_BAD_ARG, "null argument");
    if (b->n_records < 0 || p->n_cells < 0 || p->mito_length <= 0 || b->blob_bytes < 0 || n_deletions < 0)
        return fail(h, MGATK_ERR_BAD_ARG, "negative size");
    if (p->dedup_mode < 0 || p->dedup_mode > 2) return fail(h, MGATK_ERR_BAD_ARG, "dedup_mode must be 0, 1 or 2");
    if (min_clip < 1) return fail(h, MGATK_ERR_BAD_ARG, "min_clip must be >= 1");
    if (p->max_read_extent < 1) return fail(h, MGATK_ERR_BAD_ARG, "max_read_extent must be >= 1");
    if ((clip_hist_out == nullptr) != (clip_seq_out == nullptr))
        return fail(h, MGATK_ERR_BAD_ARG, "clip_hist_out and clip_seq_out go together");
    if (n_deletions > 0 && (!left_dev || !right_dev || (p->n_cells > 0 && !counts_out)))
        return fail(h, MGATK_ERR_BAD_ARG, "null deletion array");
    if (b->n_records > 0 && (!b->pos || !b->tlen || !b->flag || !b->mapq || !b->bc_idx || !b->l_seq || !b->n_cigar || !b->blob_off))
        return fail(h, MGATK_ERR_BAD_ARG, "null batch array");
    if (b->blob_bytes > 0 && !b->blob) return fail(h, MGATK_ERR_BAD_ARG, "null blob");
    if (((uintptr_t)b->blob & 15) != 0) return fail(h, MGATK_ERR_BAD_ARG, "blob must be 16-byte aligned");
    if (p->max_read_extent > (1 << 20)) return fail(h, MGATK_ERR_EXTENT, "max_read_extent above 2^20");
    if (n_deletions > MGATK_DEL_MAX) return fail(h, MGATK_ERR_RANGE, "more than MGATK_DEL_MAX deletions");
    if (p->mito_length >= (1 << 24)) return fail(h, MGATK_ERR_RANGE, "mito_length must be below 2^24");
    if (b->n_records >= (int64_t)0x7fffff00) return fail(h, MGATK_ERR_RANGE, "at most 2^31-257 records per batch");
    const bool discover = clip_hist_out != nullptr;
    if (b->n_records == 0 || (n_deletions == 0 && !discover)) return MGATK_OK;
    CU(cudaSetDevice(h->device));
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t n = b->n_records;
    u64 bits = 32, table_max = 1024;
    while (bits < (u64)p->mito_length) bits <<= 1;
    while (table_max < 2ull * (u64)n) table_max <<= 1;
    const size_t o_byl = 256, o_byr = o_byl + align_up(kDelMax * 8), o_dl = o_byr + align_up(kDelMax * 8);
    const size_t o_dr = o_dl + align_up(kDelMax * 4), o_bitmap = o_dr + align_up(kDelMax * 4);
    const size_t o_rel = o_bitmap + align_up(bits / 8), o_table = o_rel + align_up((size_t)n * 4);
    int rc = ensure(h, h->del_scratch, o_table + (size_t)table_max * sizeof(DelEntry));
    if (rc) return rc;
    char *base = (char *)h->del_scratch.p;
    DelArgs a;
    a.b = *b; a.n_cells = p->n_cells; a.P = p->mito_length; a.extent = p->max_read_extent; a.min_mapq = p->min_mapq;
    a.dedup_mode = p->dedup_mode; a.min_clip = min_clip; a.n_del = n_deletions; a.discover = discover ? 1 : 0;
    a.bitmap_mask = (u32)(bits - 1);
    a.left = left_dev; a.right = right_dev;
    a.by_l = (int2 *)(base + o_byl); a.by_r = (int2 *)(base + o_byr); a.dl = (int32_t *)(base + o_dl); a.dr = (int32_t *)(base + o_dr);
    a.n_rel = (u32 *)base; a.rel = (u32 *)(base + o_rel); a.bitmap = (u32 *)(base + o_bitmap);
    a.table = (DelEntry *)(base + o_table); a.table_max = table_max;
    a.counts = counts_out; a.clip_hist = (u64 *)clip_hist_out; a.clip_seq = (u64 *)clip_seq_out; a.error_bits = (u64 *)error_bits_out;
    CU(cudaMemsetAsync(base, 0, 4, s));
    CU(cudaMemsetAsync(a.bitmap, 0, bits / 8, s));
    h->launches = 0;
    if (n_deletions > 0) { k_del_prep<<<1, kDelPrepThreads, 0, s>>>(a); h->launches++; }
    const int64_t want = (n + kDelThreads - 1) / kDelThreads;
    const unsigned grid = (unsigned)(want < 8 * h->sm_count ? want : 8 * h->sm_count);
    const unsigned wide = (unsigned)(8 * h->sm_count);            // passes over the relevant records: their count stays on the device
    k_del_relevance<<<grid, kDelThreads, 0, s>>>(a);
    h->launches++;
    if (p->dedup_mode != MGATK_DEDUP_NONE) {
        k_del_clear<<<wide, kDelThreads, 0, s>>>(a);
        k_del_insert<<<wide, kDelThreads, 0, s>>>(a);
        k_del_min<<<grid, kDelThreads, 0, s>>>(a);
        h->launches += 3;
    }
    k_del_count<<<wide, kDelThreads, 0, s>>>(a);
    h->launches++;
    CU(cudaGetLastError());
    return MGATK_OK;
}

int mgatk_louvain_host(int32_t n, const int64_t *indptr, const int32_t *indices, const double *weights, double resolution,
                       int32_t *labels_out, int32_t *n_levels_out) {
    if (n < 0 || !n_levels_out || !(resolution > 0.0) || !std::isfinite(resolution)) return MGATK_ERR_BAD_ARG;
    *n_levels_out = 0;
    if (n == 0) return MGATK_OK;
    if (!indptr || !labels_out) return MGATK_ERR_BAD_ARG;
    if (indptr[0] != 0) return MGATK_ERR_BAD_ARG;
    for (int32_t i = 0; i < n; i++)
        if (indptr[i + 1] < indptr[i]) return MGATK_ERR_BAD_ARG;
    const int64_t nnz = indptr[n];
    if (nnz > 0 && (!indices || !weights)) return MGATK_ERR_BAD_ARG;
    if (nnz >= ((int64_t)1 << 31)) return MGATK_ERR_RANGE;
    for (int64_t e = 0; e < nnz; e++)
        if (indices[e] < 0 || indices[e] >= n || !(weights[e] >= 0.0) || !std::isfinite(weights[e])) return MGATK_ERR_BAD_ARG;
    try {
        LouvainGraph g;
        g.indptr.assign(indptr, indptr + n + 1);
        g.indices.assign(indices, indices + nnz);
        g.weights.assign(weights, weights + nnz);
        louvain(std::move(g), resolution, labels_out, n_levels_out);
    } catch (const std::bad_alloc &) {
        return MGATK_ERR_RANGE;
    }
    return MGATK_OK;
}

int64_t mgatk_last_launch_count(const mgatk_handle *h) { return h ? h->launches : 0; }

int mgatk_last_stage_times(const mgatk_handle *h, const char **names, float *ms, int *n) {
    if (!h || !n) return MGATK_ERR_BAD_ARG;
    *n = 0;
    if (!h->events_ready) return MGATK_OK;
    for (int i = 0; i < h->n_stages; i++) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, h->ev[i], h->ev[i + 1]) != cudaSuccess) { cudaGetLastError(); break; }
        if (names) names[i] = h->stage_names[i];
        if (ms) ms[i] = t;
        *n = i + 1;
    }
    return MGATK_OK;
}

}  // extern "C"
