// K4: masked activation-guidance losses and their gradients (SURVEY.md 8(a) rows 10, 10b, 10c;
// losses.py:4-84 with patch_size = 1, evaluated by guided_stable_diffuser.py:417-434).
//
// Two parts.
//
// (1) dh_build_loss_plan - once per edit.  The correspondence list has ~6x duplicates at the 64x64 loss grid
//     (SURVEY.md "hard parts"); the plan groups it by DESTINATION cell (counting sort) and collapses equal
//     (src, dst) cell pairs into one entry with a multiplicity: a CSR over destination cells (row_ptr, 8-byte pairs)
//     for the general patch kernel, a sliced-ELL view of the same pairs for this file's kernel (dh_loss_plan.cuh),
//     plus per-cell multiplicities of the three background lists.
//
// (2) dh_guidance_loss - every denoising step.  ONE persistent launch for every layer: small CTAs (256 threads, four per
//     SM) pull work items - one 64x64 plane pair, or a few planes of a smaller layer - from a dynamic queue.  The item's
//     `cur` and `orig` planes are staged in shared memory by TMA bulk copies (cp.async.bulk + mbarrier complete_tx) that
//     thread 0 issues for the NEXT item as soon as every warp is done reading the current one, so the HBM reads overlap
//     the gradient write-out of this CTA and the arithmetic of the other CTAs of the SM.
//     Per plane
//         L_fg  = 1/(C N)  sum_pairs mult * |up(orig)[src] - up(cur)[dst]|
//         dL/dup(cur)[dst] = -1/(C N) sum_pairs mult * sign(...)
//     plus the background term.  One THREAD owns one destination cell (sliced ELL): it reads cur[dst] once, walks the
//     cell's distinct sources and keeps the INTEGER sign count in a register - no atomics, and integer addition is
//     associative, so the gradient is bit-reproducible (the reference's index_put(accumulate=True) backward is not, on
//     CUDA).  Layers smaller than the loss grid are resized bilinearly inside the box of pair cells only, and their
//     gradient is written at native resolution through the transposed resize in gather form.  Loss value and gradient
//     come out of the same pass: algorithmic traffic = read cur + read orig + write grad.  The last CTA to finish reduces
//     the per-channel partial sums in a fixed order and re-zeroes the two queue counters for the next launch.
#include "dh_common.cuh"
#include "dh_loss_plan.cuh"
#include "dh_tma.cuh"

#include <stdlib.h>
#include <string.h>

namespace dh {

// ------------------------------------------------------------------------------------------------
// plan builder: one CTA of 1024 threads
// ------------------------------------------------------------------------------------------------
constexpr int kPlanThreads = 1024;
constexpr int kPlanWarps = kPlanThreads / 32;
constexpr int kPlanTab = 1024;          // per-warp counter table: source cells lo .. lo + 1023 of one destination bucket per pass
constexpr int kLenClasses = 256;        // rows are bucketed by min(length, 255), descending (class 255 is then ranked exactly)

__global__ void __launch_bounds__(kPlanThreads) loss_plan_kernel(
    const int32_t* __restrict__ fg_src, const int32_t* __restrict__ fg_dst, int n_fg,
    const int32_t* __restrict__ bg_orig, int n_bg_orig, const int32_t* __restrict__ bg_trans, int n_bg_trans,
    const int32_t* __restrict__ bg_common, int n_bg_common, int grid, void* plan, int32_t* __restrict__ scratch) {
    extern __shared__ __align__(16) int psm[];
    __shared__ int scan_smem[33];
    const int cells = grid * grid;
    int* hist = psm;                       // cells
    int* start = psm + cells;              // cells + 1
    int* ucount = start + cells + 1;       // cells
    uint32_t* tabs = reinterpret_cast<uint32_t*>(ucount + cells);   // kPlanWarps * kPlanTab
    int32_t* bucket = scratch;             // n_fg: sources grouped by destination cell
    int32_t* uniq = scratch + n_fg;        // n_fg: per bucket, distinct sources (ascending) | multiplicity << 16
    const int tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    PlanView pv = plan_view(plan, grid, n_fg);

    for (int i = tid; i < cells; i += kPlanThreads) { hist[i] = 0; ucount[i] = 0; }
    __syncthreads();
    for (int n = tid; n < n_fg; n += kPlanThreads) atomicAdd(hist + fg_dst[n], 1);
    __syncthreads();
    // exclusive scan of hist -> start (each thread owns a contiguous run of cells)
    const int per = (cells + kPlanThreads - 1) / kPlanThreads;
    const int c0 = min(cells, tid * per), c1 = min(cells, c0 + per);
    int s = 0;
    for (int i = c0; i < c1; ++i) s += hist[i];
    int total;
    int run = block_exclusive_scan(s, scan_smem, total);
    for (int i = c0; i < c1; ++i) { start[i] = run; run += hist[i]; }
    if (tid == 0) start[cells] = total;
    __syncthreads();
    for (int i = tid; i < cells; i += kPlanThreads) hist[i] = start[i];        // cursors
    __syncthreads();
    for (int n = tid; n < n_fg; n += kPlanThreads) bucket[atomicAdd(hist + fg_dst[n], 1)] = fg_src[n];
    __syncthreads();
    // per destination cell (one warp each, all 32 warps): count the sources in a private shared-memory table that covers
    // kPlanTab consecutive source cells per pass (one pass for any rigid edit: a bucket's sources span a few grid rows),
    // then emit the distinct sources in ascending order
    {
        uint32_t* cnt = tabs + (size_t)wid * kPlanTab;
        for (int d = wid; d < cells; d += kPlanWarps) {
            const int b0 = start[d], b1 = start[d + 1];
            if (b0 == b1) continue;
            int lo = 0x7FFFFFFF, hi = -1;
            for (int k = b0 + lane; k < b1; k += 32) { const int v = bucket[k]; lo = min(lo, v); hi = max(hi, v); }
            lo = __reduce_min_sync(0xFFFFFFFFu, lo);
            hi = __reduce_max_sync(0xFFFFFFFFu, hi);
            int out = b0;
            for (int w0 = lo; w0 <= hi; w0 += kPlanTab) {
                const int w1 = min(hi, w0 + kPlanTab - 1);
                for (int i = lane; i <= w1 - w0; i += 32) cnt[i] = 0;
                __syncwarp();
                for (int k = b0 + lane; k < b1; k += 32) {
                    const int v = bucket[k];
                    if (v >= w0 && v <= w1) atomicAdd(cnt + (v - w0), 1u);
                }
                __syncwarp();
                for (int base = w0; base <= w1; base += 32) {
                    const int i = base + lane;
                    uint32_t c = i <= w1 ? cnt[i - w0] : 0u;
                    while (__any_sync(0xFFFFFFFFu, c > 0)) {
                        const unsigned b = __ballot_sync(0xFFFFFFFFu, c > 0);
                        const uint32_t m = c > 255u ? 255u : c;
                        if (c > 0) uniq[out + __popc(b & ((1u << lane) - 1u))] = (int32_t)((uint32_t)i | (m << 16));
                        c -= m;
                        out += __popc(b);
                    }
                }
                __syncwarp();
            }
            if (lane == 0) ucount[d] = out - b0;
        }
    }
    __syncthreads();
    // row_ptr = exclusive scan of the distinct-pair counts, then compact the buckets into the CSR
    s = 0;
    for (int i = c0; i < c1; ++i) s += ucount[i];
    run = block_exclusive_scan(s, scan_smem, total);
    const int n_pairs = total;
    for (int i = c0; i < c1; ++i) {
        pv.row_ptr[i] = run;
        const int b0 = start[i];
        for (int j = 0; j < ucount[i]; ++j) {
            const uint32_t e = (uint32_t)uniq[b0 + j];
            pv.pairs[run + j] = make_uint2((e & 0xFFFFu) | ((uint32_t)i << 16), e >> 16);
        }
        run += ucount[i];
    }
    if (tid == 0) pv.row_ptr[cells] = n_pairs;
    __syncthreads();

    // ---- sliced-ELL view: rows (destination cells with pairs) in descending order of their length, ties in raster order ----
    int* whist = reinterpret_cast<int*>(tabs);                       // [kPlanWarps][kLenClasses] per-warp class histograms
    int* wbase = whist + kPlanWarps * kLenClasses;                    // same shape: running output positions
    int* order = hist;                                                // row -> destination cell
    int* soff = start;                                                // slice -> first entry group
    for (int i = tid; i < kPlanWarps * kLenClasses; i += kPlanThreads) whist[i] = 0;
    __syncthreads();
    const int cpw = (cells + kPlanWarps - 1) / kPlanWarps;            // contiguous cells per warp
    for (int i = lane; i < cpw; i += 32) {
        const int cell = wid * cpw + i;
        const int k = cell < cells ? min(ucount[cell], kLenClasses - 1) : 0;
        if (k > 0) atomicAdd(whist + wid * kLenClasses + k, 1);
    }
    __syncthreads();
    {   // exclusive scan in (class descending, warp ascending) order; element j = (255 - class) * 32 + warp
        constexpr int kPer = kPlanWarps * kLenClasses / kPlanThreads;        // 8
        int cs[kPer];
        s = 0;
#pragma unroll
        for (int t = 0; t < kPer; ++t) {
            const int j = tid * kPer + t, k = kLenClasses - 1 - (j / kPlanWarps), w = j % kPlanWarps;
            cs[t] = k > 0 ? whist[w * kLenClasses + k] : 0;
            s += cs[t];
        }
        run = block_exclusive_scan(s, scan_smem, total);
#pragma unroll
        for (int t = 0; t < kPer; ++t) {
            const int j = tid * kPer + t, k = kLenClasses - 1 - (j / kPlanWarps), w = j % kPlanWarps;
            wbase[w * kLenClasses + k] = run;
            run += cs[t];
        }
    }
    const int n_rows = total;
    const int n_slices = (n_rows + 31) / 32;
    __syncthreads();
    for (int i0 = 0; i0 < cpw; i0 += 32) {      // stable placement: cells of a warp in ascending order, 32 at a time
        const int cell = wid * cpw + i0 + lane;
        const int k = (i0 + lane < cpw && cell < cells) ? min(ucount[cell], kLenClasses - 1) : 0;
        const unsigned peers = __match_any_sync(0xFFFFFFFFu, k);
        const int rank = __popc(peers & ((1u << lane) - 1u));
        if (k > 0) order[wbase[wid * kLenClasses + k] + rank] = cell;
        __syncwarp();
        if (k > 0 && rank == 0) wbase[wid * kLenClasses + k] += __popc(peers);
        __syncwarp();
    }
    __syncthreads();
    {   // the rows of class 255 (255 or more entries) lead the order in raster order: rank them by their exact length so that
        // the whole order is descending, which plan_ent_cap relies on.  Such rows need a multiplicity split or more than
        // 255 distinct sources, so there are at most n_fg / 255 of them (none in the plans of rigid edits).
        int n_big = 0;
        for (int w = 0; w < kPlanWarps; ++w) n_big += whist[w * kLenClasses + kLenClasses - 1];
        if (n_big > 1) {
            int* big = reinterpret_cast<int*>(tabs) + 2 * kPlanWarps * kLenClasses;      // (is_src below reuses it)
            for (int r = tid; r < n_big; r += kPlanThreads) big[r] = order[r];
            __syncthreads();
            for (int r = tid; r < n_big; r += kPlanThreads) {
                const int cell = big[r], len = ucount[cell];
                int rank = 0;
                for (int j = 0; j < n_big; ++j) {
                    const int lj = ucount[big[j]];
                    rank += (lj > len || (lj == len && j < r)) ? 1 : 0;
                }
                order[rank] = cell;
            }
            __syncthreads();
        }
    }
    {   // slice widths (longest row of the slice) and their exclusive scan
        int w = 0;
        if (tid < n_slices)
            for (int r = tid * 32; r < min(n_rows, tid * 32 + 32); ++r) w = max(w, (ucount[order[r]] + 3) & ~3);   // rows are padded to 4
        run = block_exclusive_scan(w, scan_smem, total);
        if (tid < n_slices) { soff[tid] = run; pv.ell_off[tid] = run; }
        if (tid == 0) { soff[n_slices] = total; pv.ell_off[n_slices] = total; }
    }
    const int n_groups = total;
    // the table must fit the space plan_layout reserved for it; if it ever does not, nothing is written to `ent` and the header
    // flags the plan as unusable (dh_loss_plan_info refuses it)
    const bool ell_fits = (size_t)n_groups * 32 <= plan_ent_cap(grid, n_fg);
    __syncthreads();
    // box of the cells that are the source or the destination of a pair (resized layers work inside it)
    __shared__ int box_sm[4];
    __shared__ int nonbin_sm;
    int* is_src = reinterpret_cast<int*>(tabs) + 2 * kPlanWarps * kLenClasses;     // cells ints behind the ELL histograms
    for (int i = tid; i < cells; i += kPlanThreads) is_src[i] = 0;
    if (tid == 0) { box_sm[0] = grid; box_sm[1] = -1; box_sm[2] = grid; box_sm[3] = -1; nonbin_sm = 0; }
    __syncthreads();
    for (int n = tid; n < n_fg; n += kPlanThreads) is_src[fg_src[n]] = 1;
    __syncthreads();
    for (int i = tid; i < cells; i += kPlanThreads)
        if (is_src[i] || ucount[i] > 0) {
            const int r = i / grid, c = i - r * grid;
            atomicMin(box_sm + 0, r); atomicMax(box_sm + 1, r); atomicMin(box_sm + 2, c); atomicMax(box_sm + 3, c);
        }
    __syncthreads();
    const int box_r0 = box_sm[0], box_r1 = box_sm[1], box_s0 = box_sm[2], box_s1 = box_sm[3];
    // distinct source cells -> slots (ascending cell order): is_src[cell] becomes slot + 1 (0 = not a source)
    s = 0;
    for (int i = c0; i < c1; ++i) s += is_src[i];
    run = block_exclusive_scan(s, scan_smem, total);
    const int n_usrc = total;
    for (int i = c0; i < c1; ++i)
        if (is_src[i]) { pv.usrc_cell[run] = (uint16_t)i; is_src[i] = ++run; }
    __syncthreads();
    for (int sl = wid; sl < (ell_fits ? n_slices : 0); sl += kPlanWarps) {
        const int r = sl * 32 + lane;
        const int cell = r < n_rows ? order[r] : -1;
        const int len = cell >= 0 ? ucount[cell] : 0;
        const int base = cell >= 0 ? pv.row_ptr[cell] : 0;
        pv.row_desc[r] = cell >= 0 ? ((uint32_t)cell | ((uint32_t)len << 16)) : 0u;
        uint32_t* dst = pv.ent + (size_t)soff[sl] * 32 + lane;
        for (int k = 0; k < len; ++k) {
            const uint2 e = pv.pairs[base + k];
            const uint32_t src = e.x & 0xFFFFu;
            dst[(size_t)k * 32] = src | ((uint32_t)(is_src[src] - 1) << 12) | (e.y << 24);
        }
        // every row is padded to a multiple of four entries with (first source, multiplicity 0): the kernel walks whole
        // groups of four without per-entry predicates
        for (int k = len; k < ((len + 3) & ~3); ++k) dst[(size_t)k * 32] = dst[0] & 0xFFFFFFu;
    }
    if (tid == 0) {
        PlanHeader h;
        h.n_pairs = n_pairs; h.n_fg = n_fg; h.n_bg_orig = n_bg_orig; h.n_bg_trans = n_bg_trans; h.n_bg_common = n_bg_common;
        h.grid = grid; h.cap = n_fg; h.reserved = 0;
        h.box_r0 = box_r0; h.box_r1 = box_r1; h.box_s0 = box_s0; h.box_s1 = box_s1;
        h.n_rows = n_rows; h.n_slices = n_slices; h.n_groups = n_groups; h.n_usrc = n_usrc;
        *pv.hdr = h;
    }
    __syncthreads();
    // background list multiplicities per cell (lists from np.nonzero never repeat a cell; generic callers may)
    int* co = psm;
    int* ct = psm + cells;
    int* cc = psm + 2 * cells;
    int* rowf = psm + 3 * cells;          // cell is a destination row
    for (int i = tid; i < 3 * cells; i += kPlanThreads) psm[i] = 0;
    for (int i = tid; i < cells; i += kPlanThreads) rowf[i] = pv.row_ptr[i + 1] > pv.row_ptr[i] ? 1 : 0;
    __syncthreads();
    for (int n = tid; n < n_bg_orig; n += kPlanThreads) atomicAdd(co + bg_orig[n], 1);
    for (int n = tid; n < n_bg_trans; n += kPlanThreads) atomicAdd(ct + bg_trans[n], 1);
    for (int n = tid; n < n_bg_common; n += kPlanThreads) atomicAdd(cc + bg_common[n], 1);
    __syncthreads();
    for (int i = tid; i < cells; i += kPlanThreads) {
        ushort4 v;
        v.x = (unsigned short)min(co[i], 65535); v.y = (unsigned short)min(ct[i], 65535);
        v.z = (unsigned short)min(cc[i], 65535); v.w = (unsigned short)(is_src[i] ? 1 : 0);
        pv.bgcnt[i] = v;
        if (co[i] > 1 || ct[i] > 1 || cc[i] > 1) nonbin_sm = 1;
    }
    // membership bits of the 16 own cells of every loss-kernel thread (cell 4 * (t + 256 k) + i <-> bit 4 k + i):
    // x = bg_orig | bg_trans << 16, y = bg_common | destination row << 16
    if (tid < 256) {
        uint32_t m_ot = 0, m_cr = 0;
        for (int k = 0; k < 4; ++k)
            for (int i = 0; i < 4; ++i) {
                const int q = 4 * (tid + k * 256) + i, b = 4 * k + i;
                if (q < cells) {
                    m_ot |= (co[q] ? 1u : 0u) << b; m_ot |= (ct[q] ? 1u : 0u) << (16 + b);
                    m_cr |= (cc[q] ? 1u : 0u) << b; m_cr |= (rowf[q] ? 1u : 0u) << (16 + b);
                }
            }
        pv.own_masks[tid] = make_uint2(m_ot, m_cr);
    }
    __syncthreads();
    // bit 0: every background multiplicity is 0 or 1; bit 1: the sliced-ELL table did not fit (the plan is unusable)
    if (tid == 0) pv.hdr->reserved = (nonbin_sm ? 0 : 1) | (ell_fits ? 0 : 2);
}

// ------------------------------------------------------------------------------------------------
// fused loss + gradient
// ------------------------------------------------------------------------------------------------
constexpr int kLossThreads = 256;
constexpr int kLossWarps = kLossThreads / 32;
#ifndef DH_LOSS_MAX_GROUPS
#define DH_LOSS_MAX_GROUPS 3
#endif
constexpr int kMaxGroups = DH_LOSS_MAX_GROUPS;   // groups of kLossThreads threads per CTA (one CTA per SM): 3 -> 80 registers per thread
constexpr int kPlaneCap = kMaxG * kMaxG;         // floats per tensor in the stage
constexpr int kStageFloats = 2 * kPlaneCap;      // [cur planes][orig planes] = 32 KB
constexpr int kOwnGroups = kPlaneCap / 4 / kLossThreads;   // float4 groups per thread at the 64x64 grid = 4
constexpr int kRowUnroll = 4;    // independent gathers in flight per thread in the row walk
constexpr int kWin = 16;      // up rows (columns) that can touch one native row (column): 2 * G / h <= 16 for h >= 8
constexpr int kMaxPlanesPerItem = 2;     // resized layers: one pair of planes per item (short items balance better)

struct ResizeLayout {   // float offsets into a group's scratch area (resized planes; the flat sign counts overlay them at 0)
    int uo, uc, gs, total;
    int cap_usrc, cap_slots;     // capacities (float2 entries) of uo and of uc / gs
};

struct FusedLayer {
    const float* cur;
    const float* orig;
    float* grad;
    int C, h, w;
    float fgw, bgw;
    const void* tab;      // LayerTab of a resized layer (NULL for layers at the loss-grid resolution)
    int item_begin;       // first item of this layer among the items of its kind (flat / resized)
    int ppi;              // planes per item
    int partial_begin;    // first channel of this layer in the partial-sum array
    int flat;
};

struct FusedParams {
    FusedLayer lv[kMaxLossLayers];
    int n_layers, G;
    int n_flat_items, n_small_items;
    PlanView pv;        // the plan's arrays (device pointers, resolved on the host)
    int n_fg, n_bg_orig, n_bg_trans, n_bg_common;
    int fg_kind;        // 0 = off, 1 = local_avg patch 1
    int bg_kind;        // 0 = off, 1 = global_avg, 2 = local_avg
    float* partial;     // [all channels][2]: fg sum, bg term
    unsigned int* counters;   // [0] work queue, [1] finished CTAs: zero on entry, re-zeroed by the last CTA
    float* loss_out;
    ResizeLayout lay;
    int scratch_floats;
    int ell_floats, ell_desc_at, ell_ent_at, ell_ent_cap;    // shared-memory copy of the sliced-ELL plan (0 = read it from global)
    int ell_slices;     // slices of the plan as the caller read them from the plan header (0 = unknown: read the header)
    int tab_floats;     // shared-memory copy of the table blob of resized layer `tab_layer` (0 = tables are read from global)
    int tab_layer;
    unsigned long long* debug;     // optional (DH_LOSS_DEBUG_BUF): per CTA {start ns, end ns, items, sm id}
};

struct WorkItem {
    int layer, c0, planes;
};

// Longest items first: the plane pairs of the resized layers (arithmetic heavy), then the 64x64 planes - the tail of the
// launch is then made of the shortest items.
__device__ __forceinline__ WorkItem decode_item(const FusedParams& p, int item) {
    const int flat = item >= p.n_small_items;
    const int idx = flat ? item - p.n_small_items : item;
    int l = -1;
#pragma unroll
    for (int i = 0; i < kMaxLossLayers; ++i)
        if (i < p.n_layers && p.lv[i].flat == flat && idx >= p.lv[i].item_begin) l = i;
    WorkItem w;
    w.layer = l;
    w.c0 = (idx - p.lv[l].item_begin) * p.lv[l].ppi;
    w.planes = min(p.lv[l].ppi, p.lv[l].C - w.c0);
    return w;
}

__device__ __forceinline__ void group_sync(int gid) { asm volatile("bar.sync %0, %1;" ::"r"(gid + 1), "n"(kLossThreads) : "memory"); }

template <int kN>
__device__ __forceinline__ void block_sum(float (&v)[kN], float (*red)[8], int gid) {
    static_assert(kN <= 8, "red holds 8 values per warp");
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int i = 0; i < kN; ++i) v[i] += __shfl_xor_sync(0xFFFFFFFFu, v[i], o);
    if (lane_id() == 0)
#pragma unroll
        for (int i = 0; i < kN; ++i) red[warp_id() & (kLossWarps - 1)][i] = v[i];
    group_sync(gid);
#pragma unroll
    for (int i = 0; i < kN; ++i) v[i] = red[lane_id() & (kLossWarps - 1)][i];
#pragma unroll
    for (int o = kLossWarps / 2; o > 0; o >>= 1)
#pragma unroll
        for (int i = 0; i < kN; ++i) v[i] += __shfl_xor_sync(0xFFFFFFFFu, v[i], o);
}

// Called by the compute warps of every CTA when the queue is empty; the last CTA reduces the per-channel partials in a
// fixed order -> loss_out[0] = total, [1+2l] = fg_l, [2+2l] = bg_l, and re-arms the counters.
template <class Cta>
__device__ void loss_finish(const FusedParams& p, float (*red)[8], unsigned int* ticket, const Cta& cta) {
    __threadfence();
    __syncthreads();                      // every group of the CTA is done
    if (threadIdx.x == 0) *ticket = atomicAdd(p.counters + 1, 1u);
    __syncthreads();
    if (*ticket != cta.count() - 1 || threadIdx.x >= kLossThreads) return;
    __threadfence();
    // the first group of the last CTA: per-channel partials -> per-layer sums, four layers (eight sums) per pass; every thread
    // adds a fixed subset of the channels in a fixed order and the block tree is fixed, so the value is reproducible bit for bit
    float total = 0.0f;
    for (int l0 = 0; l0 < p.n_layers; l0 += 4) {
        float v[8] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (l0 + j >= p.n_layers) break;
            const FusedLayer& L = p.lv[l0 + j];
            for (int c = threadIdx.x; c < L.C; c += kLossThreads) {
                v[2 * j] += __ldcg(p.partial + 2 * (L.partial_begin + c));
                v[2 * j + 1] += __ldcg(p.partial + 2 * (L.partial_begin + c) + 1);
            }
        }
        block_sum<8>(v, red, 0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (l0 + j >= p.n_layers) break;
            const FusedLayer& L = p.lv[l0 + j];
            const float fg = p.fg_kind ? v[2 * j] / (float)p.n_fg / (float)L.C : 0.0f;
            const float bg = p.bg_kind == 2 ? v[2 * j + 1] / (float)p.n_bg_common / (float)L.C : (p.bg_kind == 1 ? v[2 * j + 1] / (float)L.C : 0.0f);
            if (threadIdx.x == 0) { p.loss_out[1 + 2 * (l0 + j)] = fg; p.loss_out[2 + 2 * (l0 + j)] = bg; }
            if (p.fg_kind) total += L.fgw * fg;
            if (p.bg_kind) total += L.bgw * bg;
        }
        group_sync(0);        // `red` is reused by the next pass
    }
    if (threadIdx.x == 0) {
        p.loss_out[0] = total;
        p.counters[0] = 0u;       // every group has drawn its last item: the queue can be re-armed for the next launch
        p.counters[1] = 0u;
    }
}

__device__ __forceinline__ void st_cs_f4(float* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// Table loads with an L1 eviction priority (tables in global memory, kMem < 2): the gather tables (nat_ptr / nat_ent) are walked
// in data-dependent order by every plane pair and should stay in L1, the tap words stream through once per pair.
__device__ __forceinline__ uint4 ld_stream_u4(const uint4* p) {
    uint4 v;
    asm volatile("ld.global.L1::evict_first.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ uint2 ld_keep_u2(const uint2* p) {
    uint2 v;
    asm volatile("ld.global.L1::evict_last.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ int ld_keep_s32(const int32_t* p) {
    int v;
    asm volatile("ld.global.L1::evict_last.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// snake order of the slices over the compute warps: rounds of kLossWarps slices, every other round reversed, so that the
// descending slice widths add up to about the same per warp
__device__ __forceinline__ int slice_of(int round, int wid) {
    return round * kLossWarps + ((round & 1) ? kLossWarps - 1 - wid : wid);
}

// ---- layers smaller than the loss grid -----------------------------------------------------------------
// Per (plan, layer shape) tables, built once by loss_resize_setup_kernel into one compact blob of 32-bit words that the
// loss kernel copies to shared memory.  A resized plane is never up-sampled as a whole: the loss needs up(orig) at the
// distinct SOURCE cells and up(cur) at the DESTINATION rows only, and the gradient w.r.t. the native plane is a gather over
// the destination rows that a native cell's bilinear footprint touches:
//   src_taps[j]   the four native taps (16-bit offsets) and the two lambdas of source slot j            (uint4)
//   dst_taps[s]   the same for the destination cell of ELL row slot s                                   (uint4)
//   nat_ptr, nat_ent   CSR over native cells: (row slot, weight = wrow * wcol) of every destination row in the footprint
//   wo, wt        up^T(background multiplicities) at native resolution ('global_avg' term and its gradient)
struct TabHeader {
    int32_t n_usrc, n_slots, n_nat, h, w, hw;
    int32_t at_src_taps, at_dst_taps, at_nat_ptr, at_nat_ent, at_wo, at_wt, total_words;      // word offsets into the blob
    int32_t pad[3];
};
static_assert(sizeof(TabHeader) == 64, "the blob header is 16 words");

__host__ __device__ inline size_t tab_capacity_words(int grid) {
    const size_t cells = (size_t)grid * grid;
    // header + taps of every cell twice + nat_ptr + 4 footprint entries per destination row + wo + wt (native <= grid)
    return 16 + 4 * cells + 4 * cells + (cells + 4) + 2 * (4 * cells + 3 * cells) + 2 * cells + 64;
}

struct SetupParams {
    const void* plan;
    int plan_cap, G, h, w, fg_kind, bg_kind;
};

constexpr int kSetupThreads = 1024;

__global__ void __launch_bounds__(kSetupThreads) loss_resize_setup_kernel(const __grid_constant__ SetupParams p, uint32_t* __restrict__ blob) {
    __shared__ float tmp[kMaxNative * kMaxG];
    __shared__ int16_t slot_of_cell[kMaxG * kMaxG];
    __shared__ int ty0[kMaxG], ty1[kMaxG], tx0[kMaxG], tx1[kMaxG];
    __shared__ float tly[kMaxG], tlx[kMaxG];
    __shared__ int ylo[kMaxNative], yhi[kMaxNative], xlo[kMaxNative], xhi[kMaxNative];
    __shared__ float wrow[kMaxNative * kWin], wcol[kMaxNative * kWin];
    __shared__ int scan_smem[33];
    const int tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    const int G = p.G, h = p.h, w = p.w, hw = h * w, cells = G * G;
    const PlanView pv = plan_view(const_cast<void*>(p.plan), G, p.plan_cap);
    const int n_usrc = p.fg_kind ? pv.hdr->n_usrc : 0;
    const int n_slots = p.fg_kind ? pv.hdr->n_slices * 32 : 0;
    const float sy = (float)h / (float)G, sx = (float)w / (float)G;
    if (tid < G) {
        bilinear_tap(tid, h, sy, ty0[tid], ty1[tid], tly[tid]);
        bilinear_tap(tid, w, sx, tx0[tid], tx1[tid], tlx[tid]);
    }
    for (int i = tid; i < cells; i += kSetupThreads) slot_of_cell[i] = -1;
    __syncthreads();
    if (tid < h) {       // up rows that touch native row tid, and their weights
        // (taps with weight zero - the clamped rows at the top border have i1 = 1 with lambda = 0 - are not part of the window)
        int lo = G, hi = -1;
        for (int r = 0; r < G; ++r)
            if ((ty0[r] == tid && tly[r] < 1.0f) || (ty1[r] == tid && tly[r] > 0.0f)) { lo = min(lo, r); hi = max(hi, r); }
        hi = min(hi, lo + kWin - 1);
        ylo[tid] = lo; yhi[tid] = hi;
        for (int r = lo; r <= hi; ++r)
            wrow[tid * kWin + r - lo] = (ty0[r] == tid ? 1.0f - tly[r] : 0.0f) + (ty1[r] == tid ? tly[r] : 0.0f);
    }
    if (tid >= 64 && tid - 64 < w) {
        const int j = tid - 64;
        int lo = G, hi = -1;
        for (int s = 0; s < G; ++s)
            if ((tx0[s] == j && tlx[s] < 1.0f) || (tx1[s] == j && tlx[s] > 0.0f)) { lo = min(lo, s); hi = max(hi, s); }
        hi = min(hi, lo + kWin - 1);
        xlo[j] = lo; xhi[j] = hi;
        for (int s = lo; s <= hi; ++s)
            wcol[j * kWin + s - lo] = (tx0[s] == j ? 1.0f - tlx[s] : 0.0f) + (tx1[s] == j ? tlx[s] : 0.0f);
    }
    for (int sl = tid; sl < n_slots; sl += kSetupThreads) {
        const uint32_t d = pv.row_desc[sl];
        if (d >> 16) slot_of_cell[d & 0xFFFFu] = (int16_t)sl;
    }
    __syncthreads();
    // blob layout (compact)
    TabHeader H;
    H.n_usrc = n_usrc; H.n_slots = n_slots; H.h = h; H.w = w; H.hw = hw;
    H.at_src_taps = 16;
    H.at_dst_taps = H.at_src_taps + 4 * n_usrc;
    H.at_nat_ptr = H.at_dst_taps + 4 * n_slots;
    H.at_nat_ent = H.at_nat_ptr + (hw + 1 + 3) / 4 * 4;
    // native CSR: count, scan, fill - every native cell walks the up cells of its footprint in raster order (deterministic)
    int cnt = 0;
    int my_first = 0;
    // every thread owns a contiguous run of native cells
    const int per = (hw + kSetupThreads - 1) / kSetupThreads;
    const int n0 = min(hw, tid * per), n1 = min(hw, n0 + per);
    for (int n = n0; n < n1; ++n) {
        const int y = n / w, x = n - y * w;
        for (int r = ylo[y]; r <= yhi[y]; ++r)
            for (int s2 = xlo[x]; s2 <= xhi[x]; ++s2) cnt += slot_of_cell[r * G + s2] >= 0 ? 1 : 0;
        cnt = (cnt + 3) & ~3;       // every native cell's list is padded to a multiple of four (weight 0): unrolled gather
    }
    int total;
    my_first = block_exclusive_scan(cnt, scan_smem, total);
    H.n_nat = total;
    H.at_wo = H.at_nat_ent + (2 * total + 3) / 4 * 4;
    H.at_wt = H.at_wo + (hw + 3) / 4 * 4;
    H.total_words = H.at_wt + (hw + 3) / 4 * 4;
    H.pad[0] = H.pad[1] = H.pad[2] = 0;
    if (tid == 0) *reinterpret_cast<TabHeader*>(blob) = H;
    {
        int32_t* nat_ptr = reinterpret_cast<int32_t*>(blob + H.at_nat_ptr);
        uint2* nat_ent = reinterpret_cast<uint2*>(blob + H.at_nat_ent);
        int o = my_first;
        for (int n = n0; n < n1; ++n) {
            nat_ptr[n] = o;
            const int y = n / w, x = n - y * w;
            for (int r = ylo[y]; r <= yhi[y]; ++r)
                for (int s2 = xlo[x]; s2 <= xhi[x]; ++s2) {
                    const int sl = slot_of_cell[r * G + s2];
                    if (sl >= 0) nat_ent[o++] = make_uint2((uint32_t)sl, __float_as_uint(wrow[y * kWin + r - ylo[y]] * wcol[x * kWin + s2 - xlo[x]]));
                }
            while ((o - nat_ptr[n]) & 3) nat_ent[o++] = make_uint2(0u, 0u);      // padding: slot 0 with weight 0
        }
        if (tid == 0) nat_ptr[hw] = total;
    }
    // taps of the source slots and of the destination rows
    auto taps_of = [&](int cell) {
        const int r = cell / G, s2 = cell - r * G;
        const uint32_t y0 = (uint32_t)(ty0[r] * w), y1 = (uint32_t)(ty1[r] * w), x0 = (uint32_t)tx0[s2], x1 = (uint32_t)tx1[s2];
        return make_uint4((y0 + x0) | ((y0 + x1) << 16), (y1 + x0) | ((y1 + x1) << 16), __float_as_uint(tlx[s2]), __float_as_uint(tly[r]));
    };
    uint4* src_taps = reinterpret_cast<uint4*>(blob + H.at_src_taps);
    uint4* dst_taps = reinterpret_cast<uint4*>(blob + H.at_dst_taps);
    for (int j = tid; j < n_usrc; j += kSetupThreads) src_taps[j] = taps_of((int)pv.usrc_cell[j]);
    for (int sl = tid; sl < n_slots; sl += kSetupThreads) {
        const uint32_t d = pv.row_desc[sl];
        dst_taps[sl] = (d >> 16) ? taps_of((int)(d & 0xFFFFu)) : make_uint4(0u, 0u, 0u, 0u);
    }
    // wo / wt = up^T applied to the background multiplicities (separable, via tmp)
    for (int pass = 0; pass < 2; ++pass) {
        float* dst = reinterpret_cast<float*>(blob + (pass == 0 ? H.at_wo : H.at_wt));
        __syncthreads();
        for (int y = wid; y < h; y += kSetupThreads / 32)
            for (int s2 = lane; s2 < G; s2 += 32) {
                float a = 0.0f;
                for (int r = ylo[y]; r <= yhi[y]; ++r) {
                    const ushort4 bc = pv.bgcnt[r * G + s2];
                    a = fmaf(wrow[y * kWin + r - ylo[y]], (float)(pass == 0 ? bc.x : bc.y), a);
                }
                tmp[y * G + s2] = a;
            }
        __syncthreads();
        for (int y = wid; y < h; y += kSetupThreads / 32)
            for (int x = lane; x < w; x += 32) {
                float a = 0.0f;
                for (int s2 = xlo[x]; s2 <= xhi[x]; ++s2) a = fmaf(wcol[x * kWin + s2 - xlo[x]], tmp[y * G + s2], a);
                dst[y * w + x] = a;
            }
    }
}

struct FusedShared {
    float red[kLossWarps][8];
    float red32[32];
    float lconst[kMaxLossLayers][4];
    unsigned int ticket;
    int item, layer, c0, planes;      // the item whose planes are (being) staged, decoded by thread 0
    uint64_t full;                    // mbarrier: the stage holds `item`
};

// sum over the CTA of kN values per thread, results in every thread; fixed order (warp tree, then a tree over the warp
// partials that every warp evaluates identically) -> deterministic.  One barrier.
// One pair: acc += m |d|, cnt -= m sign(d), with t = copysign(m, d): m |d| = t d, and t is only counted when d != 0.
// The counts are integer valued floats (|sum| < 2^24, checked on the host): every partial sum is exact, so the order of
// the additions does not matter and the gradient stays bit-reproducible.
__device__ __forceinline__ void pair_term(float fm, float d, float& acc, float& cnt) {
    const float t = copysignf(fm, d);
    acc = fmaf(t, d, acc);
    if (d != 0.0f) cnt -= t;
}

// kG = 64: the loss grid of the reference; kG = 0: any grid <= 64.
// kBinary: every background multiplicity is 0 or 1 (lists from np.nonzero) -> register bit masks for the own cells.
// One CTA per SM, made of up to kMaxGroups independent GROUPS of 256 threads.  A group is what a small CTA would be - its own
// stage, scratch area, mbarrier and named barrier - but all groups of the SM share one copy of the sliced-ELL plan in shared
// memory (the pair entries are re-read for every plane; from L1 / L2 they were the dominant stall).
// kG = 64: the loss grid of the reference; kG = 0: any grid <= 64.
// kBinary: every background multiplicity is 0 or 1 (lists from np.nonzero) -> register bit masks for the own cells.
// kMem: 0 = the ELL plan and the resize tables are read from global memory (through L1), 1 = the plan is in shared memory,
// 2 = the plan and the tables of the (single) resized layer are.  A template parameter so that the accesses compile to LDS.
// kGroups: groups per CTA the kernel is compiled for.  3 (80 registers) is the general build; 4 (64 registers, 1024 threads) is
// compiled WITHOUT the resized-layer path and is used for launches whose layers all have the loss-grid resolution - which is what
// guided_inference issues with the reference's weight schedule (its only resized layer always has weight 0 and is skipped).
// Where a CTA sits among the CTAs that serve its edit: the whole grid (loss_fused_kernel; WholeGrid, dh_loss_plan.cuh) or the
// edit's share of the grid (loss_fused_batch_kernel).  The single-edit position reads blockIdx / gridDim where they are used, as a plain kernel would.
struct EditShare {
    // shared memory: first CTA of the edit, CTAs of the edit (read where used rather than held in registers: the 3-group body
    // runs at its 80-register cap, and two more live registers cost spills)
    const unsigned int* first_n;
    __device__ __forceinline__ unsigned int index() const { return blockIdx.x - first_n[0]; }
    __device__ __forceinline__ unsigned int count() const { return first_n[1]; }
};

// The body of one edit's launch.  kBatch: the edit may have no sliced-ELL table while the batch's placement is kMem >= 1 (an
// empty foreground list next to non-empty ones): its plan copy is then skipped.
template <int kG, bool kBinary, int kMem, int kGroups, bool kBatch, class Cta>
__device__ __forceinline__ void loss_fused_body(const FusedParams& p, const Cta& cta) {
    constexpr bool kHasSmall = kGroups < 4;
    extern __shared__ __align__(128) float fsm[];
    __shared__ __align__(16) FusedShared shg[kGroups];
    __shared__ __align__(8) uint64_t plan_bar;       // mbarrier: the plan copy (kMem >= 1)
    const int gid = threadIdx.x / kLossThreads, tid = threadIdx.x % kLossThreads, lane = lane_id(), wid = tid >> 5;
    FusedShared& sh = shg[gid];
#ifdef DH_LOSS_PHASE_TIMERS
    const long long dbg_clock0 = clock64();
#endif
    float* const gbase = fsm + p.ell_floats + p.tab_floats + (size_t)gid * (kStageFloats + p.scratch_floats);
    float* const st_cur = gbase;                      // the stage: [cur planes][orig planes]
    float* const st_org = gbase + kPlaneCap;
    float* const scratch = gbase + kStageFloats;
    const int n_items = p.n_flat_items + p.n_small_items;

    // Thread 0 is also the producer: it draws the next item from the queue while the current one is processed and, as soon
    // as every warp is done with the stage, issues the TMA bulk copies of the next item's planes (cp.async.bulk, completion
    // on the `full` mbarrier).  Several CTAs per SM keep HBM busy while one of them waits.
    auto stage_item = [&](int item) {
        sh.item = item;
        if (item >= n_items) {          // sentinel: the queue is empty
            mbar_arrive(&sh.full);
            return;
        }
        const WorkItem it = decode_item(p, item);
        const FusedLayer& L = p.lv[it.layer];
        sh.layer = it.layer; sh.c0 = it.c0; sh.planes = it.planes;
        const size_t off = (size_t)it.c0 * L.h * L.w;
        const uint32_t bytes = (uint32_t)(it.planes * L.h * L.w) * 4u;
        mbar_arrive_expect_tx(&sh.full, 2u * bytes);
        tma_bulk_g2s(st_cur, L.cur + off, bytes, &sh.full);
        tma_bulk_g2s(st_org, L.orig + off, bytes, &sh.full);
    };
    // The first item of every group is static (item b + n * g for group g of CTA b of n: the longest items are spread over
    // the SMs first), so its planes are on their way before anything else happens; later items are drawn from the queue.
    const int n_groups_total = (int)(cta.count() * (blockDim.x / kLossThreads));
    if (tid == 0) {
        mbar_init(&sh.full, 1);
        if (kMem && threadIdx.x == 0) mbar_init(&plan_bar, 1);
        mbar_fence_init();
        stage_item((int)(cta.index() + cta.count() * gid));
    }

    const int G = kG ? kG : p.G, GG = G * G;
    const PlanView& pv = p.pv;
    const int n_slices = p.fg_kind ? (p.ell_slices ? p.ell_slices : pv.hdr->n_slices) : 0;
    const int n_rounds = (n_slices + kLossWarps - 1) / kLossWarps;
    // the sliced-ELL plan: one copy in shared memory for all groups (kMem >= 1), else read through L1
    const uint32_t* const s_words = reinterpret_cast<const uint32_t*>(fsm);
    if (kMem && threadIdx.x == 0) {
        // three TMA bulk copies (one L2 round trip, no thread waits on a load): slice offsets (padded to 16 bytes in the plan),
        // row descriptors and entries; sizes and shared-memory offsets are the caller's (multiples of 16 bytes by construction)
        uint32_t* const s_w = reinterpret_cast<uint32_t*>(fsm);
        const uint32_t b_off = (uint32_t)p.ell_desc_at * 4u, b_desc = (uint32_t)n_slices * 128u, b_ent = (uint32_t)p.ell_ent_cap * 4u;
        mbar_arrive_expect_tx(&plan_bar, b_off + b_desc + b_ent);
        if (!kBatch || b_off) tma_bulk_g2s(s_w, pv.ell_off, b_off, &plan_bar);
        if (!kBatch || b_desc) tma_bulk_g2s(s_w + p.ell_desc_at, pv.row_desc, b_desc, &plan_bar);
        if (!kBatch || b_ent) tma_bulk_g2s(s_w + p.ell_ent_at, pv.ent, b_ent, &plan_bar);
    }
    auto ell_off_of = [&](int sl) -> int { return kMem ? (int)s_words[sl] : __ldg(pv.ell_off + sl); };
    auto row_desc_of = [&](int i) -> uint32_t { return kMem ? s_words[p.ell_desc_at + i] : __ldg(pv.row_desc + i); };
    auto entries_of = [&](int sl) -> const uint32_t* { return (kMem ? s_words + p.ell_ent_at : pv.ent) + ell_off_of(sl) * 32; };
    auto ld_ent = [&](const uint32_t* q) -> uint32_t { return kMem ? *q : __ldg(q); };
    // membership of the own cells (flat layers) in the three background lists and in the set of destination rows, as
    // 16-bit masks (bit 4k+i = cell i of group k), precomputed by the plan.  Lists that come from np.nonzero never repeat a
    // cell; if a generic caller does, the multiplicities are re-read from the plan in the (slower) general path.
    const uint2 own = pv.own_masks[tid];
    const uint32_t m_ot = own.x;                                   // low half: bg_orig, high half: bg_trans
    const uint32_t m_cr = p.fg_kind ? own.y : (own.y & 0xFFFFu);   // low half: bg_common, high half: destination rows
    // multiplicity of own cell (k, i) in list `which` (0 = bg_orig, 1 = bg_trans, 2 = bg_common)
    auto wgt = [&](int k, int i, int which) -> float {
        if (kBinary) return (float)(((which == 2 ? m_cr : m_ot) >> ((which == 1 ? 16 : 0) + 4 * k + i)) & 1u);
        const ushort4 bc = pv.bgcnt[4 * (tid + k * kLossThreads) + i];
        return (float)(which == 0 ? bc.x : which == 1 ? bc.y : bc.z);
    };
    if (tid < p.n_layers) {
        const FusedLayer& L = p.lv[tid];
        // an empty index list makes the reference's loss NaN (mean over nothing) but its gradient ZERO: scale 0, not inf
        sh.lconst[tid][0] = p.fg_kind && p.n_fg > 0 ? L.fgw / ((float)L.C * (float)p.n_fg) : 0.0f;
        sh.lconst[tid][1] = p.bg_kind == 2 && p.n_bg_common > 0 ? L.bgw / ((float)L.C * (float)p.n_bg_common) : 0.0f;
        sh.lconst[tid][2] = p.bg_kind == 1 && p.n_bg_trans > 0 ? L.bgw / ((float)L.C * (float)p.n_bg_trans) : 0.0f;
    }
    const float inv_no = 1.0f / (float)p.n_bg_orig, inv_nt = 1.0f / (float)p.n_bg_trans;

    // resized layers: two planes are processed at a time (float2 per slot), so that the index arithmetic of the resize and of
    // the pair walk is paid once per pair of planes
    const ResizeLayout& lay = p.lay;
    float2* const uo2 = reinterpret_cast<float2*>(scratch + lay.uo);     // up(orig) at the distinct source cells (slot order)
    float2* const uc2 = reinterpret_cast<float2*>(scratch + lay.uc);     // up(cur) at the destination rows (ELL row slot order)
    float2* const gs2 = reinterpret_cast<float2*>(scratch + lay.gs);     // sign counts of the destination rows
    float* const cntb = scratch;                                         // sign counts of a flat plane (overlays the above)
    // the table blob of one resized layer lives in shared memory behind the ELL plan, shared by the groups
    const uint32_t* const s_tab = reinterpret_cast<const uint32_t*>(fsm) + p.ell_floats;
    if (kMem == 2) {
        const uint32_t* g_tab = static_cast<const uint32_t*>(p.lv[p.tab_layer].tab);
        const int words = min(p.tab_floats, (int)reinterpret_cast<const TabHeader*>(g_tab)->at_wo);      // (wo / wt stay in global memory)
        for (int i = threadIdx.x; i < words / 4; i += blockDim.x)
            reinterpret_cast<uint4*>(fsm + p.ell_floats)[i] = reinterpret_cast<const uint4*>(g_tab)[i];
    }
    __syncthreads();
    if (kMem) mbar_wait(&plan_bar, 0);          // the shared-memory copy of the plan has landed

    int prev_kind = -1;          // 0 = flat, 1 = resized: kind of this group's previous item (they share the scratch area)
    int wt_layer = -1;
    float wt_reg[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    uint32_t phase = 0;
    unsigned long long dbg_t0 = 0, dbg_items = 0;
    if (p.debug && tid == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(dbg_t0));
#ifdef DH_LOSS_PHASE_TIMERS
    long long ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, ph_t = dbg_clock0;
    { const long long t_ = clock64(); ph[6] = t_ - ph_t; ph_t = t_; }
#define DH_PH(i) { const long long t_ = clock64(); ph[i] += t_ - ph_t; ph_t = t_; }
#else
#define DH_PH(i)
#endif
    for (;;) {
        int next_item = 0;
        if (tid == 0) next_item = n_groups_total + (int)atomicAdd(p.counters, 1u);     // (its latency hides behind this item's work)
        mbar_wait(&sh.full, phase);
        DH_PH(0)
        phase ^= 1;
        if (sh.item >= n_items) break;
        ++dbg_items;
        const int l = sh.layer, c0 = sh.c0, planes = sh.planes;
        const FusedLayer& L = p.lv[l];
        const float fscale = sh.lconst[l][0], lscale = sh.lconst[l][1], gscale = sh.lconst[l][2];
        if (L.flat) {
            // ------------------------------------------------------------------ a plane at the loss-grid resolution
            const int c = c0;
            // Own cells: four 128-bit groups per thread, consumed right away - background sums, and for the local
            // background term the sign of (orig - cur) as two bits per cell.
            float sums[3] = {0.0f, 0.0f, 0.0f};          // foreground sum, two background sums
            uint32_t sign_bits = 0u;          // bit 4k+i: orig > cur, bit 16+4k+i: orig < cur at own cell i of group k
            if (p.bg_kind) {
#pragma unroll
                for (int k = 0; k < kOwnGroups; ++k) {
                    const int q = 4 * (tid + k * kLossThreads);
                    if (q < GG) {
                        const float4 c4 = *reinterpret_cast<const float4*>(st_cur + q);
                        const float4 o4 = *reinterpret_cast<const float4*>(st_org + q);
                        const float cv[4] = {c4.x, c4.y, c4.z, c4.w}, ov[4] = {o4.x, o4.y, o4.z, o4.w};
                        if (p.bg_kind == 1) {
#pragma unroll
                            for (int i = 3; i >= 0; --i) {
                                if (kBinary) {      // (adding x is fmaf(1, x, s); skipping it is fmaf(0, x, s) for finite x)
                                    if ((m_ot >> (4 * k + i)) & 1u) sums[1] += ov[i];
                                    if ((m_ot >> (16 + 4 * k + i)) & 1u) sums[2] += cv[i];
                                } else {
                                    sums[1] = fmaf(wgt(k, i, 0), ov[i], sums[1]);
                                    sums[2] = fmaf(wgt(k, i, 1), cv[i], sums[2]);
                                }
                            }
                        } else {
#pragma unroll
                            for (int i = 3; i >= 0; --i) {
                                const float d = ov[i] - cv[i];
                                sums[1] = fmaf(wgt(k, i, 2), fabsf(d), sums[1]);
                                sign_bits |= (d > 0.0f ? 1u : 0u) << (4 * k + i);
                                sign_bits |= (d < 0.0f ? 1u : 0u) << (16 + 4 * k + i);
                            }
                        }
                    }
                }
            }
            // the scratch area may still be read by slow warps (sign counts of the previous plane, a resized plane's buffers)
            group_sync(gid);
            prev_kind = 0;
            // Destination rows: one thread per destination cell, its sources from the sliced-ELL plan
            for (int rd = 0; rd < n_rounds; ++rd) {
                const int sl = slice_of(rd, wid);
                if (sl >= n_slices) break;
                const uint32_t desc = row_desc_of(sl * 32 + lane);
                const int len = (int)(desc >> 16), dcell = (int)(desc & 0xFFFFu);
                const uint32_t* e_ptr = entries_of(sl) + lane;
                const float cval = st_cur[dcell];
                float cn = 0.0f;
                for (int k = 0; k < len; k += kRowUnroll) {
                    uint32_t e[kRowUnroll];
                    float o[kRowUnroll];
#pragma unroll
                    for (int u = 0; u < kRowUnroll; ++u) e[u] = ld_ent(e_ptr + (k + u) * 32);      // (rows are padded to a multiple of kRowUnroll)
#pragma unroll
                    for (int u = 0; u < kRowUnroll; ++u) o[u] = st_org[e[u] & 0xFFFu];
#pragma unroll
                    for (int u = 0; u < kRowUnroll; ++u) pair_term((float)(e[u] >> 24), o[u] - cval, sums[0], cn);   // (m = 0 in the padding: no-op)
                }
                if (len) cntb[dcell] = cn;
            }
            block_sum<3>(sums, sh.red, gid);       // (its barrier also orders the count stores and ends the reads of the stage)
            if (tid == 0) stage_item(next_item);
            float bg_term = 0.0f, bscale = 0.0f;
            if (p.bg_kind == 1) {
                const float delta = sums[1] * inv_no - sums[2] * inv_nt;
                bg_term = fabsf(delta);
                bscale = -sgn(delta) * gscale;
            } else if (p.bg_kind == 2) {
                bg_term = sums[1];
            }
            if (tid == 0) { p.partial[2 * (L.partial_begin + c)] = sums[0]; p.partial[2 * (L.partial_begin + c) + 1] = bg_term; }
            if (L.grad) {
                float* g = L.grad + (size_t)c * GG;
#pragma unroll
                for (int k = 0; k < kOwnGroups; ++k) {
                    const int q = 4 * (tid + k * kLossThreads);
                    if (q >= GG) break;
                    const float4 ci = *reinterpret_cast<const float4*>(cntb + q);     // cells that are no row hold stale data: masked
                    const float cv[4] = {ci.x, ci.y, ci.z, ci.w};
                    float v[4];
#pragma unroll
                    for (int i = 0; i < 4; ++i) v[i] = ((m_cr >> (16 + 4 * k + i)) & 1u) ? cv[i] * fscale : 0.0f;
                    if (p.bg_kind == 1) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            if (kBinary) { if ((m_ot >> (16 + 4 * k + i)) & 1u) v[i] += bscale; }
                            else v[i] = fmaf(wgt(k, i, 1), bscale, v[i]);
                        }
                    } else if (p.bg_kind == 2) {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const float sg = (float)((sign_bits >> (4 * k + i)) & 1u) - (float)((sign_bits >> (16 + 4 * k + i)) & 1u);
                            v[i] -= sg * wgt(k, i, 2) * lscale;
                        }
                    }
                    st_cs_f4(g + q, make_float4(v[0], v[1], v[2], v[3]));
                }
            }
            DH_PH(1)
        } else if constexpr (kHasSmall) {
            // ------------------------------------------------------------------ planes of a layer below the loss grid
            const int h = L.h, w = L.w, hw = h * w;
            const uint32_t* const tab = kMem == 2 ? s_tab : static_cast<const uint32_t*>(L.tab);      // (kMem 2: one resized layer)
            const TabHeader& TH = *reinterpret_cast<const TabHeader*>(tab);
            const int n_usrc = TH.n_usrc, n_slots = TH.n_slots;
            const uint4* const src_taps = reinterpret_cast<const uint4*>(tab + TH.at_src_taps);
            const uint4* const dst_taps = reinterpret_cast<const uint4*>(tab + TH.at_dst_taps);
            const int32_t* const nat_ptr = reinterpret_cast<const int32_t*>(tab + TH.at_nat_ptr);
            const uint2* const nat_ent = reinterpret_cast<const uint2*>(tab + TH.at_nat_ent);
            const float* __restrict__ two = reinterpret_cast<const float*>(static_cast<const uint32_t*>(L.tab) + TH.at_wo);   // up^T(background
            const float* __restrict__ twt = reinterpret_cast<const float*>(static_cast<const uint32_t*>(L.tab) + TH.at_wt);   // multiplicities): L1
            // under-sized buffers (or a shared-memory table copy that was cut short): poison the result, never read garbage
            const bool overflow = n_usrc > lay.cap_usrc || n_slots > lay.cap_slots || (kMem == 2 && TH.at_wo > p.tab_floats);
            if (prev_kind == 0) group_sync(gid);      // slow warps may still read the sign counts of a flat plane
            prev_kind = 1;
            if (wt_layer != l) {        // this thread's cells of up^T(bg_trans multiplicities): the same for every plane of the layer
                wt_layer = l;
#pragma unroll
                for (int i = 0; i < 4; ++i) wt_reg[i] = (p.bg_kind == 1 && tid + i * kLossThreads < hw) ? __ldg(twt + tid + i * kLossThreads) : 0.0f;
            }
            for (int pl = 0; pl < planes; pl += 2) {
                const int c = c0 + pl;
                const bool two_planes = pl + 1 < planes;   // an odd plane at the end is paired with itself, its copy is not stored
                const float* const pc0 = st_cur + pl * hw;
                const float* const po0 = st_org + pl * hw;
                const float* const pc1 = two_planes ? pc0 + hw : pc0;
                const float* const po1 = two_planes ? po0 + hw : po0;
                const bool last_pair = pl + 2 >= planes;
                if (overflow) {
                    if (tid == 0) {
                        for (int j = 0; j < (two_planes ? 2 : 1); ++j) {
                            p.partial[2 * (L.partial_begin + c + j)] = __int_as_float(0x7FC00000);
                            p.partial[2 * (L.partial_begin + c + j) + 1] = __int_as_float(0x7FC00000);
                        }
                    }
                    group_sync(gid);
                    if (last_pair && tid == 0) stage_item(next_item);
                    continue;
                }
                // up(orig) at the source slots, up(cur) at the destination rows: four taps each
                auto bilerp2 = [&](const uint4 t, const float* q0, const float* q1) {
                    const int i00 = (int)(t.x & 0xFFFFu), i01 = (int)(t.x >> 16), i10 = (int)(t.y & 0xFFFFu), i11 = (int)(t.y >> 16);
                    const float lx = __uint_as_float(t.z), ly = __uint_as_float(t.w), hx = 1.0f - lx, hy = 1.0f - ly;
                    return make_float2(hy * (hx * q0[i00] + lx * q0[i01]) + ly * (hx * q0[i10] + lx * q0[i11]),
                                       hy * (hx * q1[i00] + lx * q1[i01]) + ly * (hx * q1[i10] + lx * q1[i11]));
                };
                for (int j = tid; j < n_usrc; j += kLossThreads) uo2[j] = bilerp2(kMem == 2 ? src_taps[j] : ld_stream_u4(src_taps + j), po0, po1);
                for (int j = tid; j < n_slots; j += kLossThreads) uc2[j] = bilerp2(kMem == 2 ? dst_taps[j] : ld_stream_u4(dst_taps + j), pc0, pc1);
                float sums[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};     // per plane: foreground sum, two background sums
                if (p.bg_kind == 1) {     // background sums at native resolution: <wo, orig>, <wt, cur>
                    for (int i = tid * 4; i < hw; i += kLossThreads * 4) {
                        const float4 a = __ldg(reinterpret_cast<const float4*>(two + i)), e = __ldg(reinterpret_cast<const float4*>(twt + i));
                        const float4 b0 = *reinterpret_cast<const float4*>(po0 + i), f0 = *reinterpret_cast<const float4*>(pc0 + i);
                        const float4 b1 = *reinterpret_cast<const float4*>(po1 + i), f1 = *reinterpret_cast<const float4*>(pc1 + i);
                        sums[1] = fmaf(a.x, b0.x, fmaf(a.y, b0.y, fmaf(a.z, b0.z, fmaf(a.w, b0.w, sums[1]))));
                        sums[2] = fmaf(e.x, f0.x, fmaf(e.y, f0.y, fmaf(e.z, f0.z, fmaf(e.w, f0.w, sums[2]))));
                        sums[4] = fmaf(a.x, b1.x, fmaf(a.y, b1.y, fmaf(a.z, b1.z, fmaf(a.w, b1.w, sums[4]))));
                        sums[5] = fmaf(e.x, f1.x, fmaf(e.y, f1.y, fmaf(e.z, f1.z, fmaf(e.w, f1.w, sums[5]))));
                    }
                }
                group_sync(gid);          // (also: every warp is past the gradient gather of the previous pair, gs2 can be rewritten)
                DH_PH(2)
                for (int rd = 0; rd < n_rounds; ++rd) {
                    const int sl = slice_of(rd, wid);
                    if (sl >= n_slices) break;
                    const int slot = sl * 32 + lane;
                    const int len = (int)(row_desc_of(slot) >> 16);
                    const uint32_t* e_ptr = entries_of(sl) + lane;
                    const float2 cval = uc2[slot];
                    float cn0 = 0.0f, cn1 = 0.0f;
                    for (int k = 0; k < len; k += kRowUnroll) {
                        uint32_t e[kRowUnroll];
                        float2 o[kRowUnroll];
#pragma unroll
                        for (int u = 0; u < kRowUnroll; ++u) e[u] = ld_ent(e_ptr + (k + u) * 32);      // (rows are padded to a multiple of kRowUnroll)
#pragma unroll
                        for (int u = 0; u < kRowUnroll; ++u) o[u] = uo2[(e[u] >> 12) & 0xFFFu];
#pragma unroll
                        for (int u = 0; u < kRowUnroll; ++u) {
                            const float fm = (float)(e[u] >> 24);          // (m = 0 in the padding: no-op)
                            pair_term(fm, o[u].x - cval.x, sums[0], cn0);
                            pair_term(fm, o[u].y - cval.y, sums[3], cn1);
                        }
                    }
                    gs2[slot] = make_float2(cn0, cn1);
                }
                DH_PH(3)
                block_sum<6>(sums, sh.red, gid);
                DH_PH(4)
                if (last_pair && tid == 0) stage_item(next_item);      // every read of the staged planes is behind the barrier
                float bscale0 = 0.0f, bscale1 = 0.0f;
                {
                    float bg0 = 0.0f, bg1 = 0.0f;
                    if (p.bg_kind == 1) {
                        const float d0 = sums[1] * inv_no - sums[2] * inv_nt, d1 = sums[4] * inv_no - sums[5] * inv_nt;
                        bg0 = fabsf(d0); bg1 = fabsf(d1);
                        bscale0 = -sgn(d0) * gscale; bscale1 = -sgn(d1) * gscale;
                    }
                    if (tid == 0) {
                        p.partial[2 * (L.partial_begin + c)] = sums[0]; p.partial[2 * (L.partial_begin + c) + 1] = bg0;
                        if (two_planes) { p.partial[2 * (L.partial_begin + c + 1)] = sums[3]; p.partial[2 * (L.partial_begin + c + 1) + 1] = bg1; }
                    }
                }
                DH_PH(5)
                if (L.grad) {
                    // gradient at native resolution: every native cell gathers the sign counts of the destination rows in its
                    // bilinear footprint (weights = transposed resize), plus the background term
                    float* g0 = L.grad + (size_t)c * hw;
                    auto gather_cell = [&](int n, float wtv) {
                        float a0 = 0.0f, a1 = 0.0f;
                        const int k1 = kMem == 2 ? nat_ptr[n + 1] : ld_keep_s32(nat_ptr + n + 1);
                        for (int k = kMem == 2 ? nat_ptr[n] : ld_keep_s32(nat_ptr + n); k < k1; k += 4) {       // (lists are padded to a multiple of four)
                            uint2 ne[4];
                            float2 gv[4];
#pragma unroll
                            for (int u = 0; u < 4; ++u) ne[u] = kMem == 2 ? nat_ent[k + u] : ld_keep_u2(nat_ent + k + u);
#pragma unroll
                            for (int u = 0; u < 4; ++u) gv[u] = gs2[ne[u].x];
#pragma unroll
                            for (int u = 0; u < 4; ++u) {
                                const float wv = __uint_as_float(ne[u].y);
                                a0 = fmaf(wv, gv[u].x, a0); a1 = fmaf(wv, gv[u].y, a1);
                            }
                        }
                        a0 = fmaf(bscale0, wtv, a0 * fscale); a1 = fmaf(bscale1, wtv, a1 * fscale);
                        g0[n] = a0;
                        if (two_planes) g0[hw + n] = a1;
                    };
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (tid + i * kLossThreads < hw) gather_cell(tid + i * kLossThreads, wt_reg[i]);
                    for (int n = tid + 4 * kLossThreads; n < hw; n += kLossThreads) gather_cell(n, p.bg_kind == 1 ? __ldg(twt + n) : 0.0f);
                }
                DH_PH(7)
            }
            DH_PH(7)
        }
    }
    if (p.debug && tid == 0) {
        unsigned long long t1;
        unsigned int smid;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t1));
        asm volatile("mov.u32 %0, %smid;" : "=r"(smid));
        const int slot = cta.index() * 4 + gid;
        p.debug[4 * slot + 0] = dbg_t0; p.debug[4 * slot + 1] = t1;
        p.debug[4 * slot + 2] = dbg_items; p.debug[4 * slot + 3] = smid;
#ifdef DH_LOSS_PHASE_TIMERS
        for (int i = 0; i < 8; ++i) p.debug[4 * 1024 + 8 * slot + i] = (unsigned long long)ph[i];
#endif
    }
    loss_finish(p, shg[0].red, &shg[0].ticket, cta);
}

template <int kG, bool kBinary, int kMem, int kGroups>
__global__ void __launch_bounds__(kLossThreads * kGroups, 1) loss_fused_kernel(const __grid_constant__ FusedParams p) {
    loss_fused_body<kG, kBinary, kMem, kGroups, false>(p, WholeGrid{});
}

// Several edits in one launch: CTAs [cta_begin[e], cta_begin[e + 1]) serve edit e with that edit's parameters, exactly as a
// loss_fused_kernel launch of cta_begin[e + 1] - cta_begin[e] CTAs would (own queue, ticket, partials and loss_out; the last
// CTA of the edit reduces it and re-arms its counters).  Launch-wide: the instantiation, the group count and the shared-memory
// carve-out (ell_floats / tab_floats / scratch_floats are the maxima over the edits, so that the group bases line up).
struct FusedBatchParams {
    FusedParams edit[kMaxBatchEdits];
    int cta_begin[kMaxBatchEdits + 1];
    int n_edits;
};
static_assert(sizeof(FusedBatchParams) <= 32764, "kernel parameters are limited to 32764 bytes");

template <int kG, bool kBinary, int kMem, int kGroups>
__global__ void __launch_bounds__(kLossThreads * kGroups, 1) loss_fused_batch_kernel(const __grid_constant__ FusedBatchParams bp) {
    int e = 0;
#pragma unroll
    for (int i = 1; i < kMaxBatchEdits; ++i)
        if (i < bp.n_edits && (int)blockIdx.x >= bp.cta_begin[i]) e = i;
    __shared__ unsigned int first_n[2];
    if (threadIdx.x == 0) { first_n[0] = (unsigned int)bp.cta_begin[e]; first_n[1] = (unsigned int)(bp.cta_begin[e + 1] - bp.cta_begin[e]); }
    __syncthreads();
    const EditShare cta{first_n};
    loss_fused_body<kG, kBinary, kMem, kGroups, true>(bp.edit[e], cta);
}

struct ScaleMany {
    float* data[kMaxLossLayers];
    unsigned long long n[kMaxLossLayers];
    unsigned int block_begin[kMaxLossLayers + 1];
    int count;
};

// several tensors in one launch (autograd's backward of the fused multi-layer loss)
__global__ void __launch_bounds__(256) scale_many_kernel(const __grid_constant__ ScaleMany m, const float* __restrict__ scale) {
    const float s = *scale;
    if (s == 1.0f) return;
    int t = 0;
#pragma unroll
    for (int i = 1; i < kMaxLossLayers; ++i)
        if (i < m.count && blockIdx.x >= m.block_begin[i]) t = i;
    float* data = m.data[t];
    const size_t n = m.n[t], n4 = n / 4;
    const size_t i = (size_t)(blockIdx.x - m.block_begin[t]) * blockDim.x + threadIdx.x;
    if (i < n4) {
        float4 v = reinterpret_cast<float4*>(data)[i];
        v.x *= s; v.y *= s; v.z *= s; v.w *= s;
        reinterpret_cast<float4*>(data)[i] = v;
    }
    if (i < (n & 3)) data[n4 * 4 + i] *= s;
}

}  // namespace dh

using namespace dh;

extern "C" {

size_t dh_loss_plan_bytes(int grid, int n_fg) {
    if (grid < 1 || grid > kMaxG || n_fg < 0) return 0;
    return plan_layout(grid, n_fg).total;
}

size_t dh_loss_plan_workspace_bytes(int grid, int n_fg) {
    if (grid < 1 || grid > kMaxG || n_fg < 0) return 0;
    return sizeof(int32_t) * 2 * (size_t)(n_fg > 0 ? n_fg : 1);
}

int dh_build_loss_plan(const int32_t* fg_src, const int32_t* fg_dst, int n_fg, const int32_t* bg_orig, int n_bg_orig,
                       const int32_t* bg_trans, int n_bg_trans, const int32_t* bg_common, int n_bg_common, int grid,
                       void* plan, size_t plan_bytes, void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(plan && ws && grid >= 1 && grid <= kMaxG);
    DH_REQUIRE(n_fg >= 0 && n_bg_orig >= 0 && n_bg_trans >= 0 && n_bg_common >= 0);
    DH_REQUIRE((fg_src && fg_dst) || n_fg == 0);
    DH_REQUIRE((bg_orig || n_bg_orig == 0) && (bg_trans || n_bg_trans == 0) && (bg_common || n_bg_common == 0));
    const int cells = grid * grid;
    // 16-bit fields of the plan: the per-cell background counts (a list longer than 65535 could repeat one cell that often)
    // and the row length in row_desc (a row has at most min(n_fg, cells + n_fg / 255) entries)
    if (n_bg_orig > 65535 || n_bg_trans > 65535 || n_bg_common > 65535) return DH_ERR_UNSUPPORTED;
    if (std::min<long long>(n_fg, cells + n_fg / 255) > 65535) return DH_ERR_UNSUPPORTED;
    if (plan_bytes < dh_loss_plan_bytes(grid, n_fg) || ws_bytes < dh_loss_plan_workspace_bytes(grid, n_fg)) return DH_ERR_WORKSPACE;
    size_t smem_ints = (size_t)3 * cells + 1 + (size_t)kPlanWarps * kPlanTab;
    if (smem_ints < (size_t)4 * cells) smem_ints = (size_t)4 * cells;
    const size_t smem = sizeof(int) * smem_ints;
    static_assert(kPlanWarps * kPlanTab >= 2 * kPlanWarps * kLenClasses, "the ELL histograms live in the counter tables");
    DH_CUDA_CHECK(cudaFuncSetAttribute(loss_plan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    loss_plan_kernel<<<1, kPlanThreads, smem, as_stream(stream)>>>(fg_src, fg_dst, n_fg, bg_orig, n_bg_orig, bg_trans, n_bg_trans,
                                                                   bg_common, n_bg_common, grid, plan, static_cast<int32_t*>(ws));
    DH_LAUNCH_CHECK();
    return DH_OK;
}

static size_t loss_ws_layout(size_t channels, size_t* o_counter) {
    size_t o = (sizeof(float) * 2 * channels + 15) / 16 * 16;
    *o_counter = o; o += 16;
    return o;
}

size_t dh_guidance_loss_workspace_bytes(int n_layers, int max_channels) {
    if (n_layers < 1 || max_channels < 1) return 0;
    size_t a;
    return loss_ws_layout((size_t)n_layers * max_channels, &a);
}

size_t dh_loss_resize_tables_bytes(void) { return sizeof(uint32_t) * tab_capacity_words(kMaxG); }

int dh_build_loss_resize_tables(const void* plan, int n_fg, int grid, int h, int w, int fg_kind, int bg_kind, void* tables,
                                void* stream) {
    DH_REQUIRE(plan && tables && grid >= 1 && grid <= kMaxG && h >= 1 && w >= 1 && n_fg >= 0);
    if (h > grid || w > grid || h > kMaxNative || w > kMaxNative) return DH_ERR_UNSUPPORTED;
    if (2 * ((grid + h - 1) / h) > kWin || 2 * ((grid + w - 1) / w) > kWin) return DH_ERR_UNSUPPORTED;
    if (h * w > 65535) return DH_ERR_UNSUPPORTED;      // 16-bit tap offsets
    SetupParams sp;
    sp.plan = plan; sp.plan_cap = n_fg; sp.G = grid; sp.h = h; sp.w = w; sp.fg_kind = fg_kind; sp.bg_kind = bg_kind;
    loss_resize_setup_kernel<<<1, kSetupThreads, 0, as_stream(stream)>>>(sp, static_cast<uint32_t*>(tables));
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_loss_plan_info(const void* plan_header_host, dh_loss_plan_desc* desc) {
    DH_REQUIRE(plan_header_host && desc);
    const PlanHeader* h = static_cast<const PlanHeader*>(plan_header_host);
    if (h->reserved & 2) return DH_ERR_UNSUPPORTED;        // the builder found no room for the sliced-ELL table
    desc->n_pairs = h->n_pairs;
    desc->flags = h->reserved & 1;
    desc->box_cells = h->box_r1 >= h->box_r0 ? (h->box_r1 - h->box_r0 + 1) * (h->box_s1 - h->box_s0 + 1) : 0;
    desc->ell_slices = h->n_slices;
    desc->ell_groups = h->n_groups;
    desc->n_src_cells = h->n_usrc;
    return DH_OK;
}

// What the launch rule needs to know about one edit; prepare_edit fills it next to the edit's FusedParams.
struct EditLaunchInfo {
    int n_items;        // work items
    int ell_words;      // size of the shared-memory copy of the sliced-ELL plan (0: the plan has none)
    int tab_words;      // size of the shared-memory copy of the first resized layer's tables (0: no resized layer)
    bool tab_ok;        // that copy can be used: exactly one resized layer, 64 x 64 grid
    bool binary;        // bit 0 of the plan flags: every background multiplicity is 0 or 1
};

// developer knobs, read once per process: DH_LOSS_DEBUG_BUF (address of a device buffer for tools/k4_timeline.py),
// DH_LOSS_NO_FOUR_GROUPS, DH_LOSS_MEM (cap the shared-memory placement: 0, 1, 2), DH_LOSS_GROUPS (cap the groups per CTA)
struct LossKnobs {
    unsigned long long* debug;
    bool no_four;
    int mem_cap, groups_cap;
};
static const LossKnobs& loss_knobs() {
    static const LossKnobs knobs = [] {
        LossKnobs k;
        const char* e = getenv("DH_LOSS_DEBUG_BUF");
        k.debug = e ? reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0)) : nullptr;
        k.no_four = getenv("DH_LOSS_NO_FOUR_GROUPS") != nullptr;
        e = getenv("DH_LOSS_MEM");
        k.mem_cap = e ? atoi(e) : 99;
        e = getenv("DH_LOSS_GROUPS");
        k.groups_cap = e && atoi(e) >= 1 ? atoi(e) : 99;
        return k;
    }();
    return knobs;
}

// Validates one edit and builds its FusedParams (everything but the launch-wide shared-memory placement).  No CUDA call.
// A zero source-cell or slice count in the descriptor is read as "unknown" (budget for the whole grid), except with
// exact_if_empty for an edit without foreground pairs, whose counts are exactly zero: in a batch such an edit must not
// raise the launch-wide shared-memory maxima of the other edits.
static int prepare_edit(const dh_loss_layer* layers_host, int n_layers, int grid, const void* plan, const dh_loss_plan_desc* desc,
                        int n_fg, int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind, float* loss_out,
                        void* ws, size_t ws_bytes, bool exact_if_empty, FusedParams& fp, EditLaunchInfo& info) {
    DH_REQUIRE(desc);
    const int plan_flags = desc->flags, ell_slices = desc->ell_slices, ell_groups = desc->ell_groups;
    DH_REQUIRE(layers_host && n_layers >= 1 && n_layers <= kMaxLossLayers && loss_out && ws && plan);
    DH_REQUIRE(grid >= 1 && grid <= kMaxG);
    DH_REQUIRE(n_fg >= 0 && n_bg_orig >= 0 && n_bg_trans >= 0 && n_bg_common >= 0);
    if (bg_kind != 0 && bg_kind != 1 && bg_kind != 2) return DH_ERR_INVALID_ARGUMENT;
    if (fg_kind != 0 && fg_kind != 1) return DH_ERR_INVALID_ARGUMENT;
    memset(&fp, 0, sizeof(fp));
    const int GG = grid * grid;
    int chan = 0, first_small = -1, n_small_layers = 0;
    for (int i = 0; i < n_layers; ++i) {
        const dh_loss_layer& s = layers_host[i];
        DH_REQUIRE(s.cur && s.orig && s.channels >= 1 && s.h >= 1 && s.w >= 1);
        if (s.h > kMaxNative || s.w > kMaxNative || s.h > grid || s.w > grid) return DH_ERR_UNSUPPORTED;
        // the transposed-resize tables hold kWin up rows (columns) per native row (column): 2 * ceil(grid / h) of them are needed
        if (2 * ((grid + s.h - 1) / s.h) > kWin || 2 * ((grid + s.w - 1) / s.w) > kWin) return DH_ERR_UNSUPPORTED;
        if (((size_t)s.h * s.w) % 4 != 0) return DH_ERR_UNSUPPORTED;     // 16-byte bulk copies, 128-bit plane accesses
        if ((reinterpret_cast<uintptr_t>(s.cur) & 15) || (reinterpret_cast<uintptr_t>(s.orig) & 15) ||
            (s.grad && (reinterpret_cast<uintptr_t>(s.grad) & 15)))
            return DH_ERR_INVALID_ARGUMENT;
        const bool flat = s.h == grid && s.w == grid;
        if (!flat && (!s.resize_tables || (reinterpret_cast<uintptr_t>(s.resize_tables) & 15))) return DH_ERR_INVALID_ARGUMENT;
        FusedLayer& L = fp.lv[i];
        L.cur = s.cur; L.orig = s.orig; L.grad = s.grad;
        L.C = s.channels; L.h = s.h; L.w = s.w; L.fgw = s.fg_weight; L.bgw = s.bg_weight;
        L.tab = flat ? nullptr : s.resize_tables;
        L.flat = flat ? 1 : 0;
        L.partial_begin = chan;
        chan += s.channels;
        if (flat) {
            L.ppi = 1;
            L.item_begin = fp.n_flat_items;
            fp.n_flat_items += s.channels;
        } else {
            int ppi = kPlaneCap / (s.h * s.w);
            if (ppi > kMaxPlanesPerItem) ppi = kMaxPlanesPerItem;
            if (ppi < 1) ppi = 1;
            L.ppi = ppi;
            L.item_begin = fp.n_small_items;
            fp.n_small_items += (s.channels + ppi - 1) / ppi;
            if (bg_kind == 2) return DH_ERR_UNSUPPORTED;      // 'local_avg' on a resized layer: dh_guidance_loss_patch (patch 1)
            if (first_small < 0) first_small = i;
            ++n_small_layers;
        }
    }
    fp.n_layers = n_layers;
    fp.G = grid;
    size_t o_counter;
    if (ws_bytes < loss_ws_layout((size_t)chan, &o_counter)) return DH_ERR_WORKSPACE;
    fp.pv = plan_view(const_cast<void*>(plan), grid, n_fg);
    if (n_fg >= (1 << 24)) return DH_ERR_UNSUPPORTED;      // sign counts are integer valued floats
    fp.n_fg = n_fg; fp.n_bg_orig = n_bg_orig; fp.n_bg_trans = n_bg_trans; fp.n_bg_common = n_bg_common;
    fp.fg_kind = fg_kind; fp.bg_kind = bg_kind;
    fp.partial = static_cast<float*>(ws);
    fp.counters = reinterpret_cast<unsigned int*>(static_cast<char*>(ws) + o_counter);
    fp.loss_out = loss_out;
    fp.debug = loss_knobs().debug;
    const bool exact = exact_if_empty && n_fg == 0;
    // scratch of a group: the slot arrays of a resized plane pair, overlaid with the sign counts of a flat plane
    auto up4 = [](int v) { return (v + 3) / 4 * 4; };
    ResizeLayout& lay = fp.lay;
    int o = 0;
    if (fp.n_small_items) {
        const int n_src = fg_kind ? (desc->n_src_cells > 0 || exact ? desc->n_src_cells : GG) : 0;
        const int n_slots = fg_kind ? (ell_slices > 0 || exact ? ell_slices * 32 : GG) : 0;
        lay.cap_usrc = n_src; lay.cap_slots = n_slots;
        lay.uo = o; o += up4(2 * n_src);
        lay.uc = o; o += up4(2 * n_slots);
        lay.gs = o; o += up4(2 * n_slots);
    }
    if (fp.n_flat_items && GG > o) o = GG;
    lay.total = o;
    fp.scratch_floats = (up4(o) + 31) / 32 * 32;      // (groups stay 128-byte aligned)
    int ell_words = 0;
    if (fg_kind && ell_slices > 0 && ell_groups > 0) {
        fp.ell_desc_at = up4(ell_slices + 1);
        fp.ell_ent_at = fp.ell_desc_at + ell_slices * 32;
        fp.ell_ent_cap = ell_groups * 32;
        fp.ell_slices = ell_slices;
        ell_words = up4(fp.ell_ent_at + fp.ell_ent_cap);
        ell_words = (ell_words + 31) / 32 * 32;        // the groups' stages stay 128-byte aligned
    }
    // table blob of the first resized layer: its exact size is on the device; budget for the largest it can be given the plan
    int tab_words = 0;
    if (first_small >= 0) {
        const dh_loss_layer& sl = layers_host[first_small];
        const int n_src = fg_kind ? (desc->n_src_cells > 0 || exact ? desc->n_src_cells : GG) : 0;
        const int n_slots = fg_kind ? (ell_slices > 0 || exact ? ell_slices * 32 : GG) : 0;
        const int n_rows_max = n_slots;
        tab_words = 16 + 4 * n_src + 4 * n_slots + up4(sl.h * sl.w + 1) + up4(2 * (4 * n_rows_max + 3 * sl.h * sl.w));      // (everything in front of wo / wt; native lists padded to 4)
        tab_words = (tab_words + 31) / 32 * 32;
    }
    // (the tables of ONE resized layer fit; with several resized layers they all stay in global memory)
    fp.ell_floats = 0; fp.tab_floats = 0; fp.tab_layer = first_small >= 0 ? first_small : 0;
    info.n_items = fp.n_flat_items + fp.n_small_items;
    info.ell_words = ell_words;
    info.tab_words = tab_words;
    info.tab_ok = n_small_layers == 1 && tab_words > 0 && grid == 64;
    info.binary = (plan_flags & 1) != 0;
    return DH_OK;
}

// per-process caches of the launch geometry queries (the loss entry points run every denoising step)
struct LaunchCache {
    int sms, max_smem;
    size_t smem_attr_set[20];      // per instantiation: [0, 10) loss_fused_kernel, [10, 20) loss_fused_batch_kernel
};
static int launch_cache(LaunchCache** out) {
    static LaunchCache caches[64];          // zero-initialised; one entry per device (function attributes are per device)
    int dev = 0;
    DH_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return DH_ERR_UNSUPPORTED;
    LaunchCache& lc = caches[dev];
    if (!lc.sms) {
        DH_CUDA_CHECK(cudaDeviceGetAttribute(&lc.sms, cudaDevAttrMultiProcessorCount, dev));
        DH_CUDA_CHECK(cudaDeviceGetAttribute(&lc.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    }
    *out = &lc;
    return DH_OK;
}

struct LaunchChoice {
    int groups, mem;    // groups of kLossThreads per CTA; shared-memory placement (the kMem of the instantiation)
    int vi;             // instantiation, index into loss_variants
    size_t smem;        // dynamic shared memory per CTA
};

// The launch rule: the group count, the shared-memory placement and the instantiation for a launch whose edits need at most
// ell_words / tab_words / scratch_floats of shared memory and have n_items work items in all.
static int choose_launch(const LaunchCache& lc, int grid, bool any_small, int n_items, int ell_words, int tab_words, bool tab_ok,
                         int scratch_floats, bool binary, LaunchChoice& ch) {
    const LossKnobs& knobs = loss_knobs();
    // shared memory: [one copy of the sliced-ELL plan][per group: stage + scratch]; as many groups (<= 3) as fit, the plan copy
    // is dropped (entries then come through L1) before the group count goes below two
    const size_t group_bytes = sizeof(float) * ((size_t)kStageFloats + scratch_floats);
    const size_t static_bytes = 2304;       // FusedShared x kMaxGroups and the driver's reservation, rounded up
    const size_t budget = (size_t)lc.max_smem > static_bytes ? (size_t)lc.max_smem - static_bytes : 0;
    // preference: three groups with the plan and the tables in shared memory, then without the tables, then two groups ...
    int groups = 0, mem = 0;
    const size_t ellb = sizeof(float) * ell_words, tabb = sizeof(float) * tab_words;
    // launches without a resized layer use the 64-register build: up to four groups per SM
    const bool flat_build = !any_small && grid == 64 && !knobs.no_four;
    for (int g = std::min(flat_build ? 4 : kMaxGroups, knobs.groups_cap); g >= 1 && !groups; --g) {
        if (ell_words && tab_ok && ellb + tabb + g * group_bytes <= budget) { groups = g; mem = 2; }
        else if (ell_words && grid == 64 && ellb + g * group_bytes <= budget && g >= 2) { groups = g; mem = 1; }
        else if (g * group_bytes <= budget && (g >= 2 || !ell_words)) { groups = g; mem = 0; }
    }
    if (!groups) {
        if (group_bytes > budget) return DH_ERR_UNSUPPORTED;
        groups = 1;
    }
    if (knobs.mem_cap >= 0 && knobs.mem_cap < mem) mem = knobs.mem_cap;
    if (!(flat_build && mem == 1) && groups > kMaxGroups) groups = kMaxGroups;      // only the flat build runs four groups
    if (knobs.groups_cap < groups) groups = knobs.groups_cap;
    while (groups > 1 && lc.sms * (groups - 1) >= n_items) --groups;      // tiny problems: no idle groups
    const size_t smem = sizeof(float) * ((size_t)(mem >= 1 ? ell_words : 0) + (mem == 2 ? tab_words : 0)) + groups * group_bytes;
    if (smem > budget + static_bytes) return DH_ERR_UNSUPPORTED;
    // bit 0 of the plan flags: background multiplicities are all 0/1 (lists from np.nonzero) -> register bit masks
    const bool four = flat_build && mem == 1;      // (the flat build is instantiated with the plan in shared memory)
    // (shared-memory placement is only instantiated for the reference's 64 x 64 grid)
    ch.vi = four ? 8 + (binary ? 1 : 0) : grid == 64 ? 2 + 2 * mem + (binary ? 1 : 0) : (binary ? 1 : 0);
    ch.groups = groups;
    ch.mem = mem;
    ch.smem = smem;
    return DH_OK;
}

#define DH_LOSS_VARIANTS(K)                                                                                        \
    { K<0, false, 0, kMaxGroups>, K<0, true, 0, kMaxGroups>, K<64, false, 0, kMaxGroups>, K<64, true, 0, kMaxGroups>, \
      K<64, false, 1, kMaxGroups>, K<64, true, 1, kMaxGroups>, K<64, false, 2, kMaxGroups>, K<64, true, 2, kMaxGroups>, \
      K<64, false, 1, 4>, K<64, true, 1, 4> }

// Launches the edits bp.edit[0, n_edits) that prepare_edit filled (one grid, fg_kind and bg_kind).  One edit runs
// loss_fused_kernel with bp.edit[0] alone, the 16x smaller parameter block; several run loss_fused_batch_kernel with all of bp.
static int launch_edits(FusedBatchParams& bp, const EditLaunchInfo* info, int n_edits, int grid, void* stream) {
    int n_items = 0, ell_words = 0, tab_words = 0, scratch_floats = 0;
    bool any_small = false, tab_ok = true, binary = true;
    for (int e = 0; e < n_edits; ++e) {
        n_items += info[e].n_items;
        ell_words = std::max(ell_words, info[e].ell_words);
        tab_words = std::max(tab_words, info[e].tab_words);
        scratch_floats = std::max(scratch_floats, bp.edit[e].scratch_floats);
        any_small |= bp.edit[e].n_small_items > 0;
        tab_ok &= info[e].tab_ok;
        binary &= info[e].binary;
    }
    LaunchCache* lc = nullptr;
    int rc = launch_cache(&lc);
    if (rc != DH_OK) return rc;
    if (n_edits > lc->sms) return DH_ERR_UNSUPPORTED;      // (the one check that needs the device; no GPU has fewer than 16 SMs)
    LaunchChoice ch;
    if ((rc = choose_launch(*lc, grid, any_small, n_items, ell_words, tab_words, tab_ok, scratch_floats, binary, ch)) != DH_OK) return rc;
    // CTAs in proportion to the work items, at least one per edit, at most sms in all; no group of an edit sits idle.  For one
    // edit this is min(sms, ceil(n_items / groups)) CTAs: the whole GPU, fewer when it would leave groups without an item.
    int n_ctas = 0;
    for (int e = 0; e < n_edits; ++e) {
        FusedParams& fp = bp.edit[e];
        fp.ell_floats = ch.mem >= 1 ? ell_words : 0;
        fp.tab_floats = ch.mem == 2 ? tab_words : 0;
        fp.scratch_floats = scratch_floats;
        int share = 1 + (int)((long long)(lc->sms - n_edits) * info[e].n_items / n_items);
        const int cap = (info[e].n_items + ch.groups - 1) / ch.groups;
        if (share > cap) share = cap;
        bp.cta_begin[e] = n_ctas;
        n_ctas += share;
    }
    bp.cta_begin[n_edits] = n_ctas;
    bp.n_edits = n_edits;
    static const struct {
        void (*one[10])(const FusedParams);
        void (*many[10])(const FusedBatchParams);
    } kernels = {DH_LOSS_VARIANTS(loss_fused_kernel), DH_LOSS_VARIANTS(loss_fused_batch_kernel)};
    const bool batch = n_edits > 1;
    size_t& attr_set = lc->smem_attr_set[10 * batch + ch.vi];
    if (ch.smem > attr_set) {
        const void* kernel = batch ? (const void*)kernels.many[ch.vi] : (const void*)kernels.one[ch.vi];
        DH_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ch.smem));
        attr_set = ch.smem;
    }
    if (batch) kernels.many[ch.vi]<<<n_ctas, kLossThreads * ch.groups, ch.smem, as_stream(stream)>>>(bp);
    else kernels.one[ch.vi]<<<n_ctas, kLossThreads * ch.groups, ch.smem, as_stream(stream)>>>(bp.edit[0]);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_guidance_loss(const dh_loss_layer* layers_host, int n_layers, int grid, const void* plan, const dh_loss_plan_desc* desc,
                     int n_fg, int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind, float* loss_out,
                     void* ws, size_t ws_bytes, void* stream) {
    FusedBatchParams bp;        // (only edit[0] is filled and read)
    EditLaunchInfo info;
    const int rc = prepare_edit(layers_host, n_layers, grid, plan, desc, n_fg, n_bg_orig, n_bg_trans, n_bg_common, fg_kind, bg_kind,
                                loss_out, ws, ws_bytes, false, bp.edit[0], info);
    return rc != DH_OK ? rc : launch_edits(bp, &info, 1, grid, stream);
}

size_t dh_guidance_loss_batch_workspace_bytes(int n_edits, int n_layers, int max_channels) {
    if (n_edits < 1 || n_edits > kMaxBatchEdits) return 0;
    return (size_t)n_edits * dh_guidance_loss_workspace_bytes(n_layers, max_channels);
}

int dh_guidance_loss_batch(const dh_loss_batch_edit* edits_host, int n_edits, int grid, int fg_kind, int bg_kind, void* ws,
                           size_t ws_bytes, void* stream) {
    DH_REQUIRE(edits_host && ws && n_edits >= 1);
    if (n_edits > kMaxBatchEdits) return DH_ERR_UNSUPPORTED;
    FusedBatchParams bp;
    memset(&bp, 0, sizeof(bp));
    EditLaunchInfo info[kMaxBatchEdits];
    // edit e owns bytes [e * stride, (e + 1) * stride) of the workspace
    const size_t stride = ws_bytes / (size_t)n_edits / 16 * 16;
    for (int e = 0; e < n_edits; ++e) {
        const dh_loss_batch_edit& E = edits_host[e];
        const int rc = prepare_edit(E.layers, E.n_layers, grid, E.plan, &E.desc, E.n_fg, E.n_bg_orig, E.n_bg_trans, E.n_bg_common, fg_kind,
                                    bg_kind, E.loss_out, static_cast<char*>(ws) + e * stride, stride, true, bp.edit[e], info[e]);
        if (rc != DH_OK) return rc;
        // a descriptor that gives no sliced-ELL size for a plan with pairs: dh_guidance_loss then reads the slice count from the
        // plan and keeps the plan in global memory, but a batch may place the other edits' plans in shared memory, sized by
        // their descriptors - this edit's copy would not fit there
        if (fg_kind && E.n_fg > 0 && info[e].ell_words == 0) return DH_ERR_INVALID_ARGUMENT;
    }
    return launch_edits(bp, info, n_edits, grid, stream);
}

int dh_scale_inplace_many(float* const* data_host, const size_t* n_host, int count, const float* scale, void* stream) {
    DH_REQUIRE(data_host && n_host && scale && count >= 0 && count <= kMaxLossLayers);
    ScaleMany m;
    memset(&m, 0, sizeof(m));
    unsigned int blocks = 0;
    for (int i = 0; i < count; ++i) {
        if (!data_host[i] || n_host[i] == 0) continue;
        if (reinterpret_cast<uintptr_t>(data_host[i]) & 15) return DH_ERR_INVALID_ARGUMENT;
        const size_t threads = n_host[i] / 4 > 3 ? n_host[i] / 4 : 4;
        m.data[m.count] = data_host[i]; m.n[m.count] = n_host[i]; m.block_begin[m.count] = blocks;
        blocks += (unsigned int)((threads + 255) / 256);
        ++m.count;
    }
    if (m.count == 0) return DH_OK;
    m.block_begin[m.count] = blocks;
    scale_many_kernel<<<blocks, 256, 0, as_stream(stream)>>>(m, scale);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // extern "C"
