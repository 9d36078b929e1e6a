// Shared definitions of the K4 loss kernels: the per-edit loss plan (dh_build_loss_plan) and the bilinear taps.
#pragma once
#include "dh_common.cuh"

namespace dh {

constexpr int kMaxLossLayers = 8;
constexpr int kMaxG = 64;
constexpr int kMaxNative = 64;
constexpr int kMaxBatchEdits = 16;       // edits of one batched K4 launch (dh_guidance_loss_batch, dh_guidance_loss_patch_batch)

// The CTAs of a single-edit launch: the whole grid serves the edit (the batched kernels pass the CTA's share of its edit).
struct WholeGrid {
    __device__ __forceinline__ unsigned int index() const { return blockIdx.x; }
    __device__ __forceinline__ unsigned int count() const { return gridDim.x; }
};

struct PlanHeader {
    int32_t n_pairs, n_fg, n_bg_orig, n_bg_trans, n_bg_common, grid, cap, reserved;
    int32_t box_r0, box_r1, box_s0, box_s1;   // box (loss-grid rows / columns) of the cells that are a pair source or destination
    int32_t n_rows, n_slices, n_groups, n_usrc;  // sliced-ELL view of the pairs (below); number of distinct source cells
};
static_assert(sizeof(PlanHeader) == 64, "the host reads the first 64 bytes of a plan");

// The pairs exist in two forms.  CSR over destination cells (row_ptr, pairs) is what the general patch kernel walks.
// The patch-1 kernel uses a sliced-ELL view of the same pairs: the destination cells that have pairs ("rows") are sorted
// by their number of distinct sources (descending, ties in raster order) and cut into slices of 32 rows; lane i of a warp
// owns row 32 s + i of slice s and walks ITS entries k = 0 .. len-1 at ent[(ell_off[s] + k) * 32 + i] (coalesced, no padding
// is ever read).  One thread per destination cell: the gradient of a cell is a plain store, no atomics.
struct PlanView {
    PlanHeader* hdr;
    int32_t* row_ptr;      // cells + 1
    ushort4* bgcnt;        // cells: (count in bg_orig, bg_trans, bg_common, bit0 = cell is the source of a pair)
    uint2* pairs;          // cap entries: x = src | dst << 16, y = multiplicity (<= 255; larger ones are split)
    int32_t* ell_off;      // slices + 1: first 32-entry group of every slice
    uint32_t* row_desc;    // 32 per slice: dst cell | len << 16 (len = 0: no row)
    uint32_t* ent;         // 32 per group: src cell | src slot << 12 | multiplicity << 24 (multiplicity <= 255; slot = index in usrc_cell)
    uint16_t* usrc_cell;   // cells: the distinct source cells, ascending (resized layers up-sample one value per slot)
    uint2* own_masks;      // 256: per thread of the loss kernel, membership bits of its 16 own cells (see loss_fused_kernel)
};

__host__ __device__ inline size_t plan_ent_cap(int grid, int cap) {
    const size_t cells = (size_t)grid * grid, n = cap > 0 ? (size_t)cap : 1;
    // rows in descending order of length: sum over slices of 32 * (longest row of the slice) <= n_pairs + 32 * (longest row
    // of all); a row has at most one entry per source cell plus the entries that multiplicities > 255 are split into
    // (sum of floor((m - 1) / 255) <= n / 255) (+ the padding of every row to a multiple of four entries: at most 3 * 32 per slice)
    return n + 32 * ((n < cells ? n : cells) + n / 255 + 1) + 96 * ((cells + 31) / 32);
}

struct PlanOffsets { size_t row, bg, pairs, ell_off, row_desc, ent, usrc_cell, own_masks, total; };

__host__ __device__ inline PlanOffsets plan_layout(int grid, int cap) {
    const size_t cells = (size_t)grid * grid, slices = (cells + 31) / 32;
    PlanOffsets L;
    size_t o = sizeof(PlanHeader);
    L.row = o;      o += ((cells + 1) * sizeof(int32_t) + 15) / 16 * 16;
    L.bg = o;       o += cells * sizeof(ushort4);
    L.pairs = o;    o += ((size_t)(cap > 0 ? cap : 1) * sizeof(uint2) + 15) / 16 * 16;
    L.ell_off = o;  o += ((slices + 1) * sizeof(int32_t) + 15) / 16 * 16;
    L.row_desc = o; o += slices * 32 * sizeof(uint32_t);
    L.ent = o;      o += (plan_ent_cap(grid, cap) * sizeof(uint32_t) + 15) / 16 * 16;
    L.usrc_cell = o; o += (cells * sizeof(uint16_t) + 15) / 16 * 16;
    L.own_masks = o; o += 256 * sizeof(uint2);
    L.total = o;
    return L;
}

__host__ __device__ inline PlanView plan_view(void* plan, int grid, int cap) {
    const PlanOffsets L = plan_layout(grid, cap);
    char* p = static_cast<char*>(plan);
    PlanView v;
    v.hdr = reinterpret_cast<PlanHeader*>(p);
    v.row_ptr = reinterpret_cast<int32_t*>(p + L.row);
    v.bgcnt = reinterpret_cast<ushort4*>(p + L.bg);
    v.pairs = reinterpret_cast<uint2*>(p + L.pairs);
    v.ell_off = reinterpret_cast<int32_t*>(p + L.ell_off);
    v.row_desc = reinterpret_cast<uint32_t*>(p + L.row_desc);
    v.ent = reinterpret_cast<uint32_t*>(p + L.ent);
    v.usrc_cell = reinterpret_cast<uint16_t*>(p + L.usrc_cell);
    v.own_masks = reinterpret_cast<uint2*>(p + L.own_masks);
    return v;
}

// torch area_pixel_compute_source_index (align_corners = False) for output index i
__device__ __forceinline__ void bilinear_tap(int i, int n_in, float scale, int& i0, int& i1, float& lam) {
    float src = scale * ((float)i + 0.5f) - 0.5f;
    src = src < 0.0f ? 0.0f : src;
    i0 = (int)src;
    if (i0 > n_in - 1) i0 = n_in - 1;
    i1 = i0 + (i0 < n_in - 1 ? 1 : 0);
    lam = src - (float)i0;
}

__device__ __forceinline__ float sgn(float d) { return d > 0.0f ? 1.0f : (d < 0.0f ? -1.0f : 0.0f); }

}  // namespace dh
