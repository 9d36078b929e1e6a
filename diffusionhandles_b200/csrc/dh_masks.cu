// Mask cleaning (bit-packed binary morphology), correspondence compaction, process_correspondences and
// the dense per-level source maps (SURVEY.md 8(a) rows 6, 8, 9).  All integer / bit work: bit-exact.
#include "dh_common.cuh"

namespace dh {

// ------------------------------------------------------------------------------------------------
// binary erode / dilate on row-padded bit-packed masks (bit b of word (row, w) = pixel (row, 32w+b))
// OpenCV semantics (cv2.erode / cv2.dilate with the default anchor and border): anchor = (k/2, k/2),
// dst(y,x) = op_{el(i,j) != 0} src(y + i - ay, x + j - ax); samples outside the image do not contribute.
// ------------------------------------------------------------------------------------------------
struct Element {
    uint32_t rows[32];
    int k_rows, k_cols;
    // rows with the same bit pattern form a group: shifts distribute over OR / AND, so the source rows of a group are combined
    // first and the horizontal taps are applied ONCE per group (the 10 x 10 ellipse: 4 patterns, 27 taps instead of 83)
    int n_groups;
    uint32_t group_pattern[32];
    uint32_t group_rows[32];      // bit i: element row i belongs to the group
};

__global__ void __launch_bounds__(256) morph_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                    int H, int W, int wpr, Element el, int dilate) {
    const int e = blockIdx.y;
    const int word = blockIdx.x * blockDim.x + threadIdx.x;
    if (word >= H * wpr) return;
    const int row = word / wpr, wc = word - row * wpr;
    const uint32_t* s = src + (size_t)e * H * wpr;
    const int ay = el.k_rows / 2, ax = el.k_cols / 2;
    const uint32_t fill = dilate ? 0u : 0xFFFFFFFFu;       // value of samples outside the image
    const int tail = W - (wpr - 1) * 32;                   // valid bits in the last word of a row
    const uint32_t tail_mask = tail >= 32 ? 0xFFFFFFFFu : ((1u << tail) - 1u);
    uint32_t acc = fill;
    for (int g = 0; g < el.n_groups; ++g) {
        uint32_t left = fill, mid = fill, right = fill;
        bool any = false;
        for (uint32_t rows = el.group_rows[g]; rows; rows &= rows - 1) {
            const int rr = row + (__ffs(rows) - 1) - ay;
            if (rr < 0 || rr >= H) continue;                 // rows outside the image do not contribute
            const uint32_t* r = s + (size_t)rr * wpr;
            uint32_t l = wc > 0 ? r[wc - 1] : fill;
            uint32_t m = r[wc];
            uint32_t rt = wc + 1 < wpr ? r[wc + 1] : fill;
            if (!dilate) {   // padding bits beyond W are stored as 0 but must not constrain an erosion
                if (wc == wpr - 1) m |= ~tail_mask;
                if (wc + 1 == wpr - 1) rt |= ~tail_mask;
            }
            if (dilate) { left |= l; mid |= m; right |= rt; } else { left &= l; mid &= m; right &= rt; }
            any = true;
        }
        if (!any) continue;
        for (uint32_t pat = el.group_pattern[g]; pat; pat &= pat - 1) {
            const int dx = (__ffs(pat) - 1) - ax;
            uint32_t w;
            if (dx == 0) w = mid;
            else if (dx > 0) w = __funnelshift_r(mid, right, dx);
            else w = __funnelshift_l(left, mid, -dx);
            acc = dilate ? (acc | w) : (acc & w);
        }
    }
    if (wc == wpr - 1) acc &= tail_mask;
    dst[(size_t)e * H * wpr + word] = acc;
}

// one warp per output word: bit b of word (row, w) = (mask[row][32 w + b] != 0)
__global__ void __launch_bounds__(256) pack_bits_kernel(const float* __restrict__ mask, int H, int W, int wpr, uint32_t* __restrict__ bits) {
    const int e = blockIdx.y;
    const int word = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (word >= H * wpr) return;
    const int row = word / wpr, col = (word - row * wpr) * 32 + lane_id();
    const bool on = col < W && mask[(size_t)e * H * W + (size_t)row * W + col] != 0.0f;
    const uint32_t b = __ballot_sync(0xFFFFFFFFu, on);
    if (lane_id() == 0) bits[(size_t)e * H * wpr + word] = b;
}

__global__ void __launch_bounds__(256) unpack_bits_kernel(const uint32_t* __restrict__ bits, int n_words, uint8_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_words * 32) return;
    out[i] = (bits[i >> 5] >> (i & 31)) & 1u;
}

// ------------------------------------------------------------------------------------------------
// correspondences: ordered compaction of the visible foreground points that survive the cleaned mask
// ------------------------------------------------------------------------------------------------
constexpr int kCorrTile = 1024;      // foreground points per tile (small tiles: the block scans are latency bound)
constexpr int kCorrThreads = kCorrTile / 4;

__device__ __forceinline__ bool corr_keep(const int32_t* pix, const uint32_t* winner, const uint32_t* cleaned,
                                          int e, int j, int P, int W, int wpr, int H, int stride, int& q) {
    q = pix[(size_t)e * stride + P + j];
    if (q < 0) return false;
    if (winner[(size_t)e * P + q] != (uint32_t)(P + j)) return false;
    const int row = q / W, col = q - row * W;
    return (cleaned[(size_t)e * H * wpr + row * wpr + (col >> 5)] >> (col & 31)) & 1u;
}

__global__ void __launch_bounds__(kCorrThreads) corr_count_kernel(const int32_t* __restrict__ pix, const uint32_t* __restrict__ winner,
                                                          const int32_t* __restrict__ n_fg, const uint32_t* __restrict__ cleaned,
                                                          int H, int W, int wpr, int stride, int ntiles, int32_t* __restrict__ tile_counts) {
    __shared__ int warp_sums[32];
    const int e = blockIdx.y, tile = blockIdx.x, P = H * W;
    const int n = n_fg[e];
    if (tile * kCorrTile >= n) {          // (the grid covers P points, an edit has n_fg << P)
        if (threadIdx.x == 0) tile_counts[e * ntiles + tile] = 0;
        return;
    }
    int c = 0;
    const int j0 = tile * kCorrTile + threadIdx.x * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int q;
        if (j0 + i < n && corr_keep(pix, winner, cleaned, e, j0 + i, P, W, wpr, H, stride, q)) ++c;
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if (lane_id() == 0) warp_sums[warp_id()] = c;
    __syncthreads();
    if (warp_id() == 0) {
        int s = __reduce_add_sync(0xFFFFFFFFu, lane_id() < (int)(blockDim.x >> 5) ? warp_sums[lane_id()] : 0);
        if (lane_id() == 0) tile_counts[e * ntiles + tile] = s;
    }
}

__global__ void __launch_bounds__(kCorrThreads) corr_emit_kernel(const int32_t* __restrict__ pix, const uint32_t* __restrict__ winner,
                                                         const int32_t* __restrict__ fg_index, const int32_t* __restrict__ n_fg,
                                                         const uint32_t* __restrict__ cleaned, int H, int W, int wpr, int stride,
                                                         int ntiles, const int32_t* __restrict__ tile_counts,
                                                         int64_t* __restrict__ corr, int32_t* __restrict__ n_corr) {
    __shared__ int scan_smem[33];
    __shared__ int base_smem;
    const int e = blockIdx.y, tile = blockIdx.x, P = H * W;
    const int n = n_fg[e];
    if (tile * kCorrTile >= n && tile != ntiles - 1) return;      // nothing to emit (the last tile still publishes the count)
    int part = 0;
    const int t_end = min(tile, (n + kCorrTile - 1) / kCorrTile);  // tiles beyond the edit's points hold zeros
    for (int t = threadIdx.x; t < t_end; t += blockDim.x) part += tile_counts[e * ntiles + t];
    int tot;
    block_exclusive_scan(part, scan_smem, tot);
    if (threadIdx.x == 0) base_smem = tot;
    __syncthreads();
    const int base = base_smem;
    const int j0 = tile * kCorrTile + threadIdx.x * 4;
    bool k[4];
    int q[4];
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        k[i] = j0 + i < n && corr_keep(pix, winner, cleaned, e, j0 + i, P, W, wpr, H, stride, q[i]);
        c += k[i];
    }
    int total;
    int pos = base + block_exclusive_scan(c, scan_smem, total);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!k[i]) continue;
        const int src = fg_index[(size_t)e * P + j0 + i];
        longlong4 v;   // [x_src, y_src, x_dst, y_dst], utils.py:111-113
        v.x = src % W; v.y = src / W; v.z = q[i] % W; v.w = q[i] / W;
        *reinterpret_cast<longlong4*>(corr + ((size_t)e * P + pos) * 4) = v;
        ++pos;
    }
    if (tile == ntiles - 1 && threadIdx.x == 0) n_corr[e] = base + total;
}

// ------------------------------------------------------------------------------------------------
// process_correspondences (guided_stable_diffuser.py:490-584), one CTA
// ------------------------------------------------------------------------------------------------
constexpr int kMaxGridCells = 128 * 128;

__global__ void __launch_bounds__(1024) process_corr_kernel(const int64_t* __restrict__ corr, int n_corr, int img_res, int grid,
                                                            int bg_erosion, int32_t* __restrict__ fg_src, int32_t* __restrict__ fg_dst,
                                                            int32_t* __restrict__ bg, int32_t* __restrict__ bg_orig,
                                                            int32_t* __restrict__ bg_trans, int32_t* __restrict__ counts) {
    extern __shared__ uint8_t sm[];
    __shared__ int scan_smem[33];
    const int cells = grid * grid;
    uint8_t* mo = sm;                  // bg_mask_orig
    uint8_t* mt = sm + cells;          // bg_mask_trans
    uint8_t* t0 = sm + 2 * cells;      // erosion scratch
    uint8_t* t1 = sm + 3 * cells;
    const int r = img_res / grid;
    for (int i = threadIdx.x; i < cells; i += blockDim.x) { mo[i] = 1; mt[i] = 1; }
    __syncthreads();
    // bounds filter (:509-514) + integer down-sampling (:526-527), duplicates kept, order kept
    int base = 0;
    for (int n0 = 0; n0 < n_corr; n0 += blockDim.x) {
        const int n = n0 + threadIdx.x;
        bool ok = false;
        int s = 0, d = 0;
        if (n < n_corr) {
            const longlong4 v = *reinterpret_cast<const longlong4*>(corr + (size_t)n * 4);
            ok = v.z >= 0 && v.z < img_res && v.w >= 0 && v.w < img_res;
            if (ok) {
                long long sx = v.x / r, sy = v.y / r;
                sx = sx < 0 ? 0 : (sx >= grid ? grid - 1 : sx);   // the reference would raise; stay in bounds
                sy = sy < 0 ? 0 : (sy >= grid ? grid - 1 : sy);
                s = (int)sy * grid + (int)sx;
                long long dx = v.z / r, dy = v.w / r;
                dx = dx >= grid ? grid - 1 : dx;
                dy = dy >= grid ? grid - 1 : dy;
                d = (int)dy * grid + (int)dx;
            }
        }
        int total;
        const int pos = base + block_exclusive_scan(ok ? 1 : 0, scan_smem, total);
        if (ok) {
            fg_src[pos] = s; fg_dst[pos] = d;
            mo[s] = 0; mt[d] = 0;
        }
        base += total;
    }
    __syncthreads();
    // scipy.ndimage.binary_erosion(iterations=n): 3x3 cross, border_value = 0
    for (int it = 0; it < bg_erosion; ++it) {
        for (int i = threadIdx.x; i < cells; i += blockDim.x) {
            const int y = i / grid, x = i - y * grid;
            const bool in = y > 0 && y < grid - 1 && x > 0 && x < grid - 1;
            t0[i] = in ? (mo[i] & mo[i - grid] & mo[i + grid] & mo[i - 1] & mo[i + 1]) : 0;
            t1[i] = in ? (mt[i] & mt[i - grid] & mt[i + grid] & mt[i - 1] & mt[i + 1]) : 0;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < cells; i += blockDim.x) { mo[i] = t0[i]; mt[i] = t1[i]; }
        __syncthreads();
    }
    // np.nonzero lists, row-major (:541-543)
    int nb = 0, nbo = 0, nbt = 0;
    for (int i0 = 0; i0 < cells; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        const bool o = i < cells && mo[i], t = i < cells && mt[i];
        int total;
        int pos = nb + block_exclusive_scan((o && t) ? 1 : 0, scan_smem, total);
        if (o && t) bg[pos] = i;
        nb += total;
        pos = nbo + block_exclusive_scan(o ? 1 : 0, scan_smem, total);
        if (o) bg_orig[pos] = i;
        nbo += total;
        pos = nbt + block_exclusive_scan(t ? 1 : 0, scan_smem, total);
        if (t) bg_trans[pos] = i;
        nbt += total;
    }
    if (threadIdx.x == 0) {
        counts[0] = base; counts[1] = nb; counts[2] = nbo; counts[3] = nbt; counts[4] = 0;
    }
}

// ------------------------------------------------------------------------------------------------
// dense per-level source maps: all levels of a stack in one pass
// ------------------------------------------------------------------------------------------------
constexpr int kMaxMapLevels = 8;
struct MapLevels {
    int n_levels, img_res;
    int side[kMaxMapLevels];
    int cell_begin[kMaxMapLevels + 1];      // prefix sums of side^2
    size_t map_begin[kMaxMapLevels];        // offset (ints) of level l inside the map buffer: B * cell_begin[l]
};

__global__ void __launch_bounds__(256) dense_maps_scatter_kernel(const int64_t* __restrict__ corr, const int32_t* __restrict__ n_corr,
                                                                 int corr_stride_rows, const __grid_constant__ MapLevels lv,
                                                                 int32_t* __restrict__ maps) {
    const int e = blockIdx.y;
    const int n_e = min(n_corr[e], corr_stride_rows);     // a count above the capacity would read the next edit's rows
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < n_e; n += gridDim.x * blockDim.x) {
        const longlong4 v = *reinterpret_cast<const longlong4*>(corr + ((size_t)e * corr_stride_rows + n) * 4);
        // rows with a coordinate outside the image (never produced by dh_correspondences; a caller's own list might) are ignored
        if ((unsigned long long)v.x >= (unsigned long long)lv.img_res || (unsigned long long)v.y >= (unsigned long long)lv.img_res ||
            (unsigned long long)v.z >= (unsigned long long)lv.img_res || (unsigned long long)v.w >= (unsigned long long)lv.img_res)
            continue;
#pragma unroll
        for (int l = 0; l < kMaxMapLevels; ++l) {
            if (l >= lv.n_levels) break;
            const int side = lv.side[l], r = lv.img_res / side;
            const int d = (int)(v.w / r) * side + (int)(v.z / r);
            int32_t* cell = maps + lv.map_begin[l] + (size_t)e * side * side + d;
            // the map only ever decreases, so a plain (possibly stale) read can only over-estimate it: skipping when n is not
            // below it is conservative.  Coarse levels have hundreds of correspondences per cell - almost all of them skip.
            if (n < __ldcg(cell)) atomicMin(cell, n);
        }
    }
}

// one thread per (level, destination cell): cells with a correspondence read its source; the others fall back to the first
// target pixel of the cell (raster order) that has a splat winner - almost always the very first one, the background covers
// the image - so a sequential scan per thread beats a cooperative one by keeping 32x more cells in flight
__global__ void __launch_bounds__(256) dense_maps_finalize_kernel(const int64_t* __restrict__ corr, int corr_stride_rows,
                                                                  const int32_t* __restrict__ winner_src,
                                                                  const __grid_constant__ MapLevels lv, int32_t* __restrict__ maps) {
    const int e = blockIdx.y;
    const int gcell = blockIdx.x * blockDim.x + threadIdx.x;
    if (gcell >= lv.cell_begin[lv.n_levels]) return;
    int l = 0;
#pragma unroll
    for (int i = 1; i < kMaxMapLevels; ++i)
        if (i < lv.n_levels && gcell >= lv.cell_begin[i]) l = i;
    const int side = lv.side[l], img_res = lv.img_res, r = img_res / side, cell = gcell - lv.cell_begin[l];
    int32_t* m = maps + lv.map_begin[l] + (size_t)e * side * side + cell;
    const int first = *m;
    int res = -1;
    if (first < 0x7F000000) {
        const longlong4 v = *reinterpret_cast<const longlong4*>(corr + ((size_t)e * corr_stride_rows + first) * 4);
        res = (int)(v.y / r) * side + (int)(v.x / r);
    } else if (winner_src) {
        const int cy = cell / side, cx = cell - cy * side;
        const int32_t* ws = winner_src + (size_t)e * img_res * img_res + (size_t)(cy * r) * img_res + cx * r;
        for (int dy = 0; dy < r && res < 0; ++dy) {
            const int32_t* row = ws + (size_t)dy * img_res;
            for (int dx = 0; dx < r; ++dx) {
                const int s_ = __ldg(row + dx);
                if (s_ >= 0) { res = ((s_ / img_res) / r) * side + (s_ % img_res) / r; break; }
            }
        }
    }
    *m = res;
}

}  // namespace dh

using namespace dh;

static int make_element(const uint32_t* rows_host, int k_rows, int k_cols, Element* el) {
    if (!rows_host || k_rows < 1 || k_rows > 32 || k_cols < 1 || k_cols > 32) return DH_ERR_INVALID_ARGUMENT;
    for (int i = 0; i < 32; ++i) el->rows[i] = i < k_rows ? rows_host[i] : 0u;
    el->k_rows = k_rows;
    el->k_cols = k_cols;
    el->n_groups = 0;
    for (int i = 0; i < 32; ++i) { el->group_pattern[i] = 0u; el->group_rows[i] = 0u; }
    for (int i = 0; i < k_rows; ++i) {
        const uint32_t pat = k_cols >= 32 ? el->rows[i] : (el->rows[i] & ((1u << k_cols) - 1u));
        if (!pat) continue;
        int g = 0;
        while (g < el->n_groups && el->group_pattern[g] != pat) ++g;
        if (g == el->n_groups) el->group_pattern[el->n_groups++] = pat;
        el->group_rows[g] |= 1u << i;
    }
    return DH_OK;
}

extern "C" {

int dh_morph_pass(const uint32_t* src_bits, uint32_t* dst_bits, int B, int H, int W, const uint32_t* element_rows_host,
                  int k_rows, int k_cols, int dilate, void* stream) {
    DH_REQUIRE(src_bits && dst_bits && src_bits != dst_bits && B >= 1 && H >= 1 && W >= 1);
    Element el;
    int rc = make_element(element_rows_host, k_rows, k_cols, &el);
    if (rc != DH_OK) return rc;
    const int wpr = (W + 31) / 32;
    dim3 grid((H * wpr + 255) / 256, B);
    morph_kernel<<<grid, 256, 0, as_stream(stream)>>>(src_bits, dst_bits, H, W, wpr, el, dilate ? 1 : 0);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_mask_clean(const uint32_t* target_bits, uint32_t* cleaned_bits, uint32_t* tmp_bits, int B, int H, int W,
                  const uint32_t* close_rows_host, int close_k, const uint32_t* open_rows_host, int open_k, void* stream) {
    DH_REQUIRE(target_bits && cleaned_bits && tmp_bits && cleaned_bits != tmp_bits);
    // CLOSE = dilate then erode, OPEN = erode then dilate (cv2.morphologyEx, depth_transform.py:318-321)
    int rc = dh_morph_pass(target_bits, tmp_bits, B, H, W, close_rows_host, close_k, close_k, 1, stream);
    if (rc) return rc;
    rc = dh_morph_pass(tmp_bits, cleaned_bits, B, H, W, close_rows_host, close_k, close_k, 0, stream);
    if (rc) return rc;
    rc = dh_morph_pass(cleaned_bits, tmp_bits, B, H, W, open_rows_host, open_k, open_k, 0, stream);
    if (rc) return rc;
    return dh_morph_pass(tmp_bits, cleaned_bits, B, H, W, open_rows_host, open_k, open_k, 1, stream);
}

int dh_pack_mask_bits(const float* mask, int B, int H, int W, uint32_t* bits, void* stream) {
    DH_REQUIRE(mask && bits && B >= 1 && H >= 1 && W >= 1);
    const int wpr = (W + 31) / 32;
    dim3 grid((H * wpr + 7) / 8, B);
    pack_bits_kernel<<<grid, 256, 0, as_stream(stream)>>>(mask, H, W, wpr, bits);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_unpack_bits(const uint32_t* bits, int n_words_total, uint8_t* out_u8, void* stream) {
    DH_REQUIRE(bits && out_u8 && n_words_total >= 1);
    unpack_bits_kernel<<<(n_words_total * 32 + 255) / 256, 256, 0, as_stream(stream)>>>(bits, n_words_total, out_u8);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_correspondences(const int32_t* pix, const uint32_t* winner, const int32_t* fg_index, const int32_t* n_fg,
                       const uint32_t* cleaned_bits, int B, int H, int W, int stride_points, int64_t* corr, int32_t* n_corr,
                       void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(pix && winner && fg_index && n_fg && cleaned_bits && corr && n_corr && ws && B >= 1 && H >= 1 && W >= 1);
    const int P = H * W;
    const int ntiles = (P + kCorrTile - 1) / kCorrTile;
    if (ws_bytes < sizeof(int32_t) * (size_t)B * ntiles) return DH_ERR_WORKSPACE;
    int32_t* tile_counts = static_cast<int32_t*>(ws);
    const int wpr = (W + 31) / 32;
    dim3 grid(ntiles, B);
    cudaStream_t st = as_stream(stream);
    corr_count_kernel<<<grid, kCorrThreads, 0, st>>>(pix, winner, n_fg, cleaned_bits, H, W, wpr, stride_points, ntiles, tile_counts);
    DH_LAUNCH_CHECK();
    corr_emit_kernel<<<grid, kCorrThreads, 0, st>>>(pix, winner, fg_index, n_fg, cleaned_bits, H, W, wpr, stride_points, ntiles,
                                            tile_counts, corr, n_corr);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_process_correspondences(const int64_t* corr, int n_corr, int img_res, int grid, int bg_erosion, int32_t* fg_src,
                               int32_t* fg_dst, int32_t* bg, int32_t* bg_orig, int32_t* bg_trans, int32_t* counts, void* stream) {
    DH_REQUIRE(n_corr >= 0 && (corr || n_corr == 0) && fg_src && fg_dst && bg && bg_orig && bg_trans && counts);
    DH_REQUIRE(grid >= 1 && grid * grid <= kMaxGridCells && img_res >= grid && bg_erosion >= 0);
    const size_t smem = 4 * (size_t)grid * grid;
    if (smem > 48 * 1024)
        DH_CUDA_CHECK(cudaFuncSetAttribute(process_corr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    process_corr_kernel<<<1, 1024, smem, as_stream(stream)>>>(corr, n_corr, img_res, grid, bg_erosion, fg_src, fg_dst, bg,
                                                              bg_orig, bg_trans, counts);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_dense_source_maps(const int64_t* corr, const int32_t* n_corr, int corr_stride_rows, const int32_t* winner_src, int B,
                         int img_res, const int* sides_host, int n_levels, int32_t* maps, void* stream) {
    DH_REQUIRE(corr && n_corr && maps && sides_host && B >= 1 && n_levels >= 1 && n_levels <= kMaxMapLevels);
    DH_REQUIRE(corr_stride_rows >= 1);
    MapLevels lv;
    memset(&lv, 0, sizeof(lv));
    lv.n_levels = n_levels; lv.img_res = img_res;
    int cells = 0;
    for (int l = 0; l < n_levels; ++l) {
        const int side = sides_host[l];
        DH_REQUIRE(side >= 1 && img_res >= side && img_res % side == 0);
        lv.side[l] = side; lv.cell_begin[l] = cells; lv.map_begin[l] = (size_t)B * cells;
        cells += side * side;
    }
    lv.cell_begin[n_levels] = cells;
    cudaStream_t st = as_stream(stream);
    DH_CUDA_CHECK(cudaMemsetAsync(maps, 0x7F, sizeof(int32_t) * (size_t)B * cells, st));
    int gx = (corr_stride_rows + 255) / 256;
    if (gx > 64) gx = 64;                         // grid-stride: the capacity is P rows, the lists are ~10x shorter
    dense_maps_scatter_kernel<<<dim3(gx, B), 256, 0, st>>>(corr, n_corr, corr_stride_rows, lv, maps);
    DH_LAUNCH_CHECK();
    dense_maps_finalize_kernel<<<dim3((cells + 255) / 256, B), 256, 0, st>>>(corr, corr_stride_rows, winner_src, lv, maps);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // extern "C"
