/*
 * dh_b200.h - C ABI of libdiffhandles_b200.so: the B200-native (sm_100a) implementation of the
 * DiffusionHandles activation-lifting / 3D-warp hot path.
 *
 * The reference (adobe-research/DiffusionHandles) is pure Python and has no FFI of its own; this
 * header is the boundary a maintainer would bind (ctypes stub in INTEGRATION.md).  Every entry point
 * names the reference code it replaces as file:line under /root/reference/diffhandles.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the parameter name ends in _host;
 *   - images are row-major, pixel index p = row*W + col; batches have a leading dimension B and are
 *     densely packed (edit e starts at e * per-edit element count);
 *   - functions never allocate and never synchronise; they enqueue work on `stream` (a cudaStream_t
 *     passed as void*) and return 0 or a negative dh_status.  Scratch memory comes from the caller
 *     (sizes from the *_workspace_bytes queries);
 *   - counts that only exist on the device (n_fg, n_corr) are written to device ints; the caller
 *     reads them back when it needs them on the host (the only synchronisation point of an edit);
 *   - integer / byte / index outputs are bit-exact against the reference executed with NumPy >= 2;
 *     fp32 outputs of the loss kernels are within 1e-5 relative.
 */
#ifndef DH_B200_H
#define DH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define DH_B200_ABI_VERSION 1

typedef enum dh_status {
    DH_OK = 0,
    DH_ERR_INVALID_ARGUMENT = -1,   /* null pointer, non-positive size, unsupported shape          */
    DH_ERR_UNSUPPORTED = -2,        /* valid request outside what the kernels implement            */
    DH_ERR_CUDA = -3,               /* a CUDA runtime call failed; see dh_last_cuda_error()        */
    DH_ERR_WORKSPACE = -4           /* workspace too small                                          */
} dh_status;

/* Pinhole camera: fp32 intrinsics and their fp32 inverse, row-major 3x3.
 * guided_stable_diffuser.py:129-153 (get_depth_intrinsics), depth_transform.py:595 (linalg.inv). */
typedef struct dh_camera {
    float k[9];
    float kinv[9];
} dh_camera;

/* Rigid transform of the foreground, already reduced to what the kernel consumes:
 * axis = fp32 axis / ||axis||, cos_t/sin_t = cos/sin(radians(angle)) in fp64, t = translation.
 * depth_transform.py:497-531 (transform_point_cloud). */
typedef struct dh_rigid {
    float axis[3];
    float _pad;
    double cos_t;
    double sin_t;
    double t[3];
} dh_rigid;

/* One level of an activation stack: NCHW fp32, C planes of h*w.  `in`/`out` point at edit 0; edit e
 * is at in + e*C*h*w.  `src_map` is int32[B][h*w]: source cell of every destination cell, -1 = none. */
typedef struct dh_warp_level {
    const float* in;
    float* out;
    const int32_t* src_map;
    int32_t channels;
    int32_t hw;
} dh_warp_level;

const char* dh_status_string(int status);
int dh_abi_version(void);
/* cudaError_t of the last failing CUDA call made by this library on the calling thread. */
int dh_last_cuda_error(void);
/* Multiprocessor count and compute capability of the current device (for grid sizing / checks). */
int dh_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- pixel grid: torch.linspace(start, end, steps) on CPU, depth_transform.py:623-628 (HOST) ---- */
int dh_linspace_f32_host(float start, float end, int steps, float* out_host);

/* ---- row 2: depth_to_world_coords, depth_transform.py:589-641 -------------------------------------
 * depth (B,H,W) fp32 -> points (B,H,W,3) fp32, identity extrinsics; xs (W), ys (H) = pixel grid. */
int dh_unproject(const float* depth, int B, int H, int W, const dh_camera* cam_host,
                 const float* xs, const float* ys, float* points, void* stream);

/* ---- row 3': transform_points, depth_transform.py:439-459 (torch fp32 variant, tolerance 1e-5) ----
 * points (N,3) fp32; centroid = mean of the given points; angle in degrees. ws: dh_transform_points_workspace_bytes. */
size_t dh_transform_points_workspace_bytes(int N);
int dh_transform_points(const float* points, int N, float angle_degrees, const float* axis_host3,
                        const float* translation_host3, float* out, void* ws, size_t ws_bytes, void* stream);

/* ---- per-edit scratch for the fused pc path (rows 2-6) ------------------------------------------- */
size_t dh_edit_workspace_bytes(int B, int H, int W);

/* ---- row 3: transform_point_cloud, depth_transform.py:461-533 -----------------------------------------
 * points (N,3) fp32, mask (N) fp32 (non-zero = selected): Rodrigues rotation about the fp32 sequential centroid of
 * the selected points + translation, applied to ALL N points -> out (N,3) fp64; centroid float[3]; n_masked int32. */
size_t dh_transform_point_cloud_workspace_bytes(int N);
int dh_transform_point_cloud(const float* points, const float* mask, int N, const dh_rigid* rigid_host, double* out,
                             float* centroid, int32_t* n_masked, void* ws, size_t ws_bytes, void* stream);

/* ---- row 5 (projection only): points (N,3) fp64 -> pix, zkey;  depth_transform.py:666-687 --------- */
int dh_project_points(const double* points, int N, int H, int W, const dh_camera* cam_host,
                      int32_t* pix, uint64_t* zkey, int32_t* u, int32_t* v, void* stream);

/* ---- K1 + K2 of a batch of edits in one call (what transform_depth_pc runs, depth_transform.py:226-306) ----------
 * The points of edit e, in the reference's order:
 *   points 0..P-1   = unprojected bg_depth pixels (raster order),
 *   points P..P+n-1 = unprojected depth pixels under fg_mask (non-zero = foreground), rotated about
 *                     their fp32 sequential centroid and translated (fp64), raster order of the source.
 * Per-point outputs sit at the point's index (capacity 2*P per edit): pix int32 (v*W+u, -1 = z is NaN), zkey uint64
 * (order-preserving bits of the fp64 z); optional points_out double[2P][3] (debug, may be NULL).  Per edit: fg_index int32[P]
 * (source pixel of fg point j), n_fg int32, centroid float[3], and the splat outputs of dh_splat_resolve with fg_start = P.
 * rigid_host: B structs on the host.
 * Same results as dh_splat_zbuffer + dh_splat_resolve over the generic pixel / key of every point, bit for bit, in seven
 * launches and without memsets: with the library's pinhole camera a background point provably keeps its pixel, so the
 * z-buffer is initialised with the background keys (float4 loads, 128-bit stores), the fp64 transform / projection runs for
 * the foreground points only, and a background pixel resolves itself.  Background depths that are zero, infinite or of absurd
 * magnitude, and any camera / image outside that class, take the generic per-point path inside the same kernels.
 * pix / zkey: (B, 2P) - filled for the foreground points (index P + j); the background half only when points_out != NULL
 * (debug: the generic projection of every background point).  inv_minmax as in dh_splat_resolve (may be NULL). */
int dh_edit_splat(const float* depth, const float* bg_depth, const float* fg_mask, int B, int H, int W,
                  const dh_camera* cam_host, const dh_rigid* rigid_host, const float* xs, const float* ys,
                  int32_t* pix, uint64_t* zkey, int32_t* fg_index, int32_t* n_fg, float* centroid, double* points_out,
                  uint64_t* zbuf, uint32_t* winner, float* depth_map, uint8_t* target_mask, uint32_t* target_bits,
                  int32_t* winner_src, float* inv_minmax, void* ws, size_t ws_bytes, void* stream);

/* ---- multi-object edits: dh_edit_splat with K disjoint foreground objects, each with its own rigid transform -------------
 * labels uint8[B][P]: 0 = background, k + 1 = object k (1 <= K <= 16); it must be non-zero exactly where fg_mask is, which
 * stays the union of the objects.  The points are those of dh_edit_splat over the union (foreground point j = the j-th union
 * pixel in raster order); point j belongs to the object of its pixel, fg_object uint8[B][P] records it (0..K-1), and it is
 * rotated about the fp32 sequential centroid of ITS object's points (raster order) and moved by its object's transform.
 * rigid_host: B*K structs on the host, edit-major (rigid_host[b*K + k]), uploaded with one copy; centroid float[B][K][3]
 * (NaN for an object without pixels, whose transform is then unused).  Everything else as dh_edit_splat; with K = 1 the
 * outputs are those of dh_edit_splat bit for bit.  ws: dh_edit_objects_workspace_bytes(B, H, W) (any K). */
size_t dh_edit_objects_workspace_bytes(int B, int H, int W);
int dh_edit_splat_objects(const float* depth, const float* bg_depth, const float* fg_mask, const uint8_t* labels, int B, int K,
                          int H, int W, const dh_camera* cam_host, const dh_rigid* rigid_host, const float* xs, const float* ys,
                          int32_t* pix, uint64_t* zkey, int32_t* fg_index, uint8_t* fg_object, int32_t* n_fg, float* centroid,
                          double* points_out, uint64_t* zbuf, uint32_t* winner, float* depth_map, uint8_t* target_mask,
                          uint32_t* target_bits, int32_t* winner_src, float* inv_minmax, void* ws, size_t ws_bytes, void* stream);

/* ---- K2, row 5: deterministic z-buffer splat, depth_transform.py:689-712 ---------------------------
 * winner[q] = argmin over {i : pix_i = q} of (z_i, i).  Two 64/32-bit atomicMin passes (z bits, then
 * point index among the points that tie on z) - exact for fp64 depths.
 * n_points: device int32[B] (number of valid points per edit) or NULL -> every edit has n_max points.
 * zbuf uint64[B][P], winner uint32[B][P] (0xFFFFFFFF = empty).  stride_points = per-edit capacity. */
int dh_splat_zbuffer(const int32_t* pix, const uint64_t* zkey, const int32_t* n_points, int n_fixed,
                     int n_max, int stride_points, int B, int P,
                     uint64_t* zbuf, uint32_t* winner, void* stream);

/* ---- K2 epilogue, rows 5-6: depth_transform.py:714-747, :283-306 ----------------------------------
 * depth_map fp32 (+inf = empty), target_mask uint8 {0,1} = winner is a foreground point,
 * target_bits = the same mask bit-packed (bit b of word w = pixel 32*w+b), winner_src int32 = source
 * pixel of the winner (bg point p -> p, fg point -> fg_index), -1 = empty; inv_minmax float[B][2] =
 * min/max of 1/depth_map (for normalize_depth).  Foreground points are those with index >= fg_start
 * (pc path: fg_start = P) or, if point_mask != NULL, those with point_mask[i] != 0. */
int dh_splat_resolve(const uint64_t* zbuf, const uint32_t* winner, int B, int H, int W,
                     int fg_start, const uint8_t* point_mask, const int32_t* fg_index, int stride_points,
                     float* depth_map, uint8_t* target_mask, uint32_t* target_bits, int32_t* winner_src,
                     float* inv_minmax, void* stream);

/* visible[i] = is_fg(i) && winner[pix_i] == i   (depth_transform.py:701-711, masked_point_visible_mask) */
int dh_splat_visible(const int32_t* pix, const uint32_t* winner, const int32_t* n_points, int n_fixed, int n_max,
                     int stride_points, int B, int P, int fg_start, const uint8_t* point_mask,
                     uint8_t* visible, void* stream);

/* normalize_depth(1/depth_map): 255*(x-min)/(max-min) in fp32, depth_transform.py:15-28, :289-293.
 * bounds: device float[B][2] (min,max).  dh_inv_minmax computes them from a depth image. */
int dh_inv_minmax(const float* depth, int B, int P, float* inv_minmax, void* stream);
int dh_disparity(const float* depth, int B, int P, const float* bounds, float* disparity, void* stream);

/* ---- row 6: mask cleaning, depth_transform.py:308-321 ---------------------------------------------
 * One binary erode/dilate pass on bit-packed masks with an arbitrary structuring element of at most
 * 32x32 (element rows as bit masks, bit j = column j; OpenCV anchor (k/2,k/2), border ignored). */
int dh_morph_pass(const uint32_t* src_bits, uint32_t* dst_bits, int B, int H, int W,
                  const uint32_t* element_rows_host, int k_rows, int k_cols, int dilate, void* stream);
/* cleaned = OPEN_open(CLOSE_close(target)); tmp = scratch of the same size. */
int dh_mask_clean(const uint32_t* target_bits, uint32_t* cleaned_bits, uint32_t* tmp_bits, int B, int H, int W,
                  const uint32_t* close_rows_host, int close_k, const uint32_t* open_rows_host, int open_k, void* stream);
int dh_unpack_bits(const uint32_t* bits, int n_words_total, uint8_t* out_u8, void* stream);
/* float mask (B,H,W), non-zero = set -> row-padded bit planes uint32[B][H][ceil(W/32)] */
int dh_pack_mask_bits(const float* mask, int B, int H, int W, uint32_t* bits, void* stream);

/* ---- row 6: correspondences, depth_transform.py:299-343 -------------------------------------------
 * For fg point j (raster order of the source): keep iff visible and cleaned[pix]; emits int64 (n,4)
 * rows [x_src, y_src, x_dst, y_dst] in reference order.  corr has capacity P rows per edit.
 * ws: int32[B * ceil(P / 1024)] tile counts. */
int dh_correspondences(const int32_t* pix, const uint32_t* winner, const int32_t* fg_index, const int32_t* n_fg,
                       const uint32_t* cleaned_bits, int B, int H, int W, int stride_points,
                       int64_t* corr, int32_t* n_corr, void* ws, size_t ws_bytes, void* stream);

/* ---- row 8: process_correspondences, guided_stable_diffuser.py:490-584 ----------------------------
 * corr int64 (n,4) -> cell lists on the grid x grid latent grid (reference: 64).  Outputs (device):
 * fg_src/fg_dst int32[n_valid] cell ids (y*grid+x) with multiplicity, bg / bg_orig / bg_trans cell id
 * lists (row-major nonzero order), counts int32[5] = {n_valid, n_bg, n_bg_orig, n_bg_trans, 0}. */
int dh_process_correspondences(const int64_t* corr, int n_corr, int img_res, int grid, int bg_erosion,
                               int32_t* fg_src, int32_t* fg_dst, int32_t* bg, int32_t* bg_orig, int32_t* bg_trans,
                               int32_t* counts, void* stream);

/* ---- row 9: dense per-level source maps ------------------------------------------------------------
 * src_map[q] = source cell of the lowest-n correspondence whose destination cell is q; cells without
 * one fall back (if winner_src != NULL) to the first target pixel of the cell (raster order) that has
 * a splat winner; else -1.
 * All levels of a stack in one pass (the correspondences are read once): sides_host[l] = cells per side of level l
 * (HOST array); maps = one buffer of B * sum(side_l^2) ints, level-major (level l starts at B * sum_{k<l} side_k^2,
 * inside it edit-major: B maps of side_l^2 cells).
 * corr = B lists of corr_stride_rows rows; n_corr[e] above corr_stride_rows counts as corr_stride_rows.  Rows with a
 * coordinate outside [0, img_res) are ignored. */
int dh_dense_source_maps(const int64_t* corr, const int32_t* n_corr, int corr_stride_rows, const int32_t* winner_src,
                         int B, int img_res, const int* sides_host, int n_levels, int32_t* maps, void* stream);

/* ---- K3, row 9: the activation warp ----------------------------------------------------------------
 * list form : out[c][n] = in[c][idx[n]]            (losses.py:46-47, :80)
 * dense form: out[c][q] = map[q] >= 0 ? in[c][map[q]] : 0, for every level of a stack, B edits.
 * The dense kernel stages 16 KB chunks of the source planes in shared memory with TMA bulk copies
 * (cp.async.bulk + mbarrier) and writes 128-bit rows.
 * Indices outside [0, hw) - negative or too large - give 0 and are never dereferenced (the reference's tensor indexing
 * would raise IndexError for them; a kernel cannot, so it stays memory safe instead).
 * Pointers need only fp32 / int32 alignment; a level whose pointers are not 16-byte aligned takes the generic path.
 * The dense form checks every level before its first launch, so a rejected call writes no output. */
int dh_warp_gather_list(const float* in, int C, int hw, const int32_t* idx, int n, float* out, void* stream);
int dh_warp_gather_dense(const dh_warp_level* levels_host, int n_levels, int B, void* stream);

/* ---- K4, rows 10/10b/10c: masked guidance losses + gradients, losses.py:4-84 -----------------------
 * One fused pass per layer: loss value and dL/d(cur) (native resolution, bilinear-transposed).
 * fg_kind: 0 = no foreground term, 1 = local_avg (patch 1) over the (src,dst) cell pairs;
 * bg_kind: 0 = no background term, 1 = global_avg (bg_orig / bg_trans lists), 2 = local_avg (bg_common).
 * Empty lists give NaN like the reference (mean over an empty set). */
typedef struct dh_loss_layer {
    const float* cur;       /* (C,h,w) current activations                    */
    const float* orig;      /* (C,h,w) recorded activations (this timestep)   */
    float* grad;            /* (C,h,w) out: weighted dL/dcur (may be NULL)    */
    int32_t channels, h, w;
    float fg_weight, bg_weight;
    const void* resize_tables;   /* dh_build_loss_resize_tables output when (h,w) != (grid,grid), else NULL */
} dh_loss_layer;

/* Loss plan, built once per edit from the process_correspondences lists (int32 cell ids y*grid+x): the
 * foreground pairs grouped by destination cell with duplicates collapsed into multiplicities, and the per-cell
 * multiplicities of the three background lists.  grid <= 64.  plan / ws sizes from the two queries.
 * DH_ERR_UNSUPPORTED for a background list longer than 65535 entries, or an n_fg that could give one destination cell more
 * than 65535 entries (16-bit plan fields). */
size_t dh_loss_plan_bytes(int grid, int n_fg);
size_t dh_loss_plan_workspace_bytes(int grid, int n_fg);
int dh_build_loss_plan(const int32_t* fg_src, const int32_t* fg_dst, int n_fg,
                       const int32_t* bg_orig, int n_bg_orig, const int32_t* bg_trans, int n_bg_trans,
                       const int32_t* bg_common, int n_bg_common, int grid,
                       void* plan, size_t plan_bytes, void* ws, size_t ws_bytes, void* stream);

/* Per-(plan, layer shape) tables of a layer smaller than the loss grid: bilinear taps, the transposed-resize weights,
 * up^T(background multiplicities) and the active box.  Built once per edit and layer shape, reused every step. */
size_t dh_loss_resize_tables_bytes(void);
int dh_build_loss_resize_tables(const void* plan, int n_fg, int grid, int h, int w, int fg_kind, int bg_kind,
                                void* tables, void* stream);

size_t dh_guidance_loss_workspace_bytes(int n_layers, int max_channels);
/* What the launcher needs to know about a plan; filled from a HOST copy of the first 64 bytes of the plan. */
typedef struct dh_loss_plan_desc {
    int32_t n_pairs;       /* distinct (src, dst) cell pairs                                                     */
    int32_t box_cells;     /* cells of the box that contains every pair cell                                      */
    int32_t flags;         /* bit 0: every background multiplicity is 0 or 1 (bit-mask instantiation)             */
    int32_t ell_slices;    /* size of the sliced-ELL pair table: slices of 32 destination rows ...                */
    int32_t ell_groups;    /* ... and groups of 32 entries (sizes its shared-memory copy)                         */
    int32_t n_src_cells;   /* distinct source cells (sizes the per-plane buffers of the resized layers)           */
} dh_loss_plan_desc;
/* DH_ERR_UNSUPPORTED when the builder flagged the plan as unusable (its sliced-ELL table did not fit the plan buffer). */
int dh_loss_plan_info(const void* plan_header_host, dh_loss_plan_desc* desc);
/* n_* are the list lengths the plan was built from (they are the means' denominators).  ONE persistent launch for all
 * layers.  `ws` must be zero-filled once before its first use; the launch leaves its queue counters zeroed again, so the
 * same workspace serves every following evaluation without a memset (one evaluation at a time per workspace).
 * 'local_avg' background terms on layers smaller than the grid are DH_ERR_UNSUPPORTED here: use dh_guidance_loss_patch. */
int dh_guidance_loss(const dh_loss_layer* layers_host, int n_layers, int grid, const void* plan, const dh_loss_plan_desc* desc,
                     int n_fg, int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind,
                     float* loss_out /* device float[1 + 2*n_layers]: total, then fg_l, bg_l */,
                     void* ws, size_t ws_bytes, void* stream);
/* Several edits in ONE launch: the dh_guidance_loss arguments of one edit (the plan descriptor by value). */
typedef struct dh_loss_batch_edit {
    const dh_loss_layer* layers;     /* HOST array of n_layers layer descriptors */
    int32_t n_layers;
    const void* plan;
    dh_loss_plan_desc desc;
    int32_t n_fg, n_bg_orig, n_bg_trans, n_bg_common;
    float* loss_out;                 /* device float[1 + 2*n_layers] of this edit */
} dh_loss_batch_edit;
/* Workspace of a batch: n_edits times dh_guidance_loss_workspace_bytes (0 outside 1 <= n_edits <= 16). */
size_t dh_guidance_loss_batch_workspace_bytes(int n_edits, int n_layers, int max_channels);
/* dh_guidance_loss for each of the n_edits edits of the HOST array edits_host, in one launch.  grid, fg_kind and bg_kind are
 * the same for every edit; every edit's results are bit-identical to a dh_guidance_loss call on that edit alone.  Each edit is
 * validated as dh_guidance_loss validates one and is rejected with the same code; edit e owns bytes [e s, (e+1) s) of `ws`,
 * s = ws_bytes / n_edits rounded down to 16, which must be large enough for that edit.  DH_ERR_INVALID_ARGUMENT for
 * n_edits < 1 or NULL arrays, DH_ERR_UNSUPPORTED for n_edits above 16 or above the SM count (callers split larger batches).
 * An edit with foreground pairs (fg_kind 1, n_fg > 0) whose descriptor gives no sliced-ELL size (ell_slices or ell_groups 0) is
 * DH_ERR_INVALID_ARGUMENT: fill the descriptor with dh_loss_plan_info.  Every check runs before any CUDA call, except the
 * comparison with the SM count, which follows the device query (it cannot fail on a GPU with 16 or more SMs).
 * `ws` is zeroed once; the launch re-arms it (one evaluation at a time per workspace).
 * No allocation, no synchronisation. */
int dh_guidance_loss_batch(const dh_loss_batch_edit* edits_host, int n_edits, int grid, int fg_kind, int bg_kind,
                           void* ws, size_t ws_bytes, void* stream);
/* The same losses with patch_size > 1 (losses.py:62-77: both maps are replaced by their local averages over the indexed
 * cells, AvgPool2d(patch, stride 1, padding patch//2) of w*f divided by that of w plus 1e-10, before the L1 difference;
 * 'global_avg' ignores the patch).  Same plan, layer descriptors (resize_tables unused) and loss_out layout as
 * dh_guidance_loss; 1 <= patch_size <= 31.  patch_size == 1 gives the dh_guidance_loss result. */
size_t dh_guidance_loss_patch_workspace_bytes(int n_layers, int max_channels);
int dh_guidance_loss_patch(const dh_loss_layer* layers_host, int n_layers, int grid, int patch_size, const void* plan,
                           int n_fg, int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind,
                           float* loss_out, void* ws, size_t ws_bytes, void* stream);
/* Workspace of a patch batch: n_edits times dh_guidance_loss_patch_workspace_bytes (0 outside 1 <= n_edits <= 16). */
size_t dh_guidance_loss_patch_batch_workspace_bytes(int n_edits, int n_layers, int max_channels);
/* dh_guidance_loss_patch for each of the n_edits edits of the HOST array edits_host: one main launch and one finish launch for
 * all of them.  grid, patch_size, fg_kind and bg_kind are the same for every edit (the descriptors' desc and the layers'
 * resize_tables are unused); every edit's results are bit-identical to a dh_guidance_loss_patch call on that edit alone, and a
 * batch of one edit runs exactly that call's kernels.  Edit e owns bytes [e s, (e+1) s) of `ws`, s = ws_bytes / n_edits
 * rounded down to 8, which must hold that edit's partial array.  Every check runs before any CUDA call: each edit is validated as
 * dh_guidance_loss_patch validates one and is rejected with the same code; DH_ERR_INVALID_ARGUMENT for n_edits < 1 or NULL
 * arrays, DH_ERR_UNSUPPORTED for n_edits above 16 (callers split larger batches).  No allocation, no synchronisation. */
int dh_guidance_loss_patch_batch(const dh_loss_batch_edit* edits_host, int n_edits, int grid, int patch_size, int fg_kind,
                                 int bg_kind, void* ws, size_t ws_bytes, void* stream);
/* grads *= *scale (device scalar) for up to 8 tensors in one launch (HOST arrays of device pointers and element counts); exits
 * early on the device when *scale == 1. */
int dh_scale_inplace_many(float* const* data_host, const size_t* n_host, int count, const float* scale, void* stream);

/* ---- 8(f) rank 1: Poisson hole fill of the edited disparity, depth_transform.py:346-363, :535-587 ----
 * Unknown pixels = mask_a XOR mask_b (cleaned ^ raw target mask; mask_b may be NULL).  Solves the masked
 * 5-point Laplace system (diag 4, known neighbours on the right-hand side) with fp64 conjugate gradients,
 * one 8-CTA cluster per edit; out = image with the unknown pixels replaced.  max_iter <= 0 -> 20000.
 * iters_out (device int32[B], may be NULL): iterations taken; NEGATIVE (-iterations - 1) when the solver stopped without
 * reaching rel_tol (iteration cap or breakdown) - the caller decides whether to warn or raise. */
size_t dh_poisson_workspace_bytes(int B, int H, int W);
int dh_poisson_fill(const float* image, const uint32_t* mask_a_bits, const uint32_t* mask_b_bits, int B, int H, int W,
                    float* out, int max_iter, double rel_tol, int32_t* iters_out, void* ws, size_t ws_bytes, void* stream);
/* Same system with a source term: right-hand side -= laplacian(lap_source) (5-point stencil, zero padding, rounded to
 * fp32) - solve_laplacian_depth, utils.py:49-102, used by DiffusionHandles.set_foreground (diffusion_handles.py:105-108). */
int dh_poisson_fill_source(const float* image, const uint32_t* mask_a_bits, const uint32_t* mask_b_bits,
                           const float* lap_source, int B, int H, int W, float* out, int max_iter, double rel_tol,
                           int32_t* iters_out, void* ws, size_t ws_bytes, void* stream);

/* ---- 8(f) rank 4: the elementwise steps of guided_inference around the U-Net (one launch each) ---------------------
 * out = latents - grad * step_size (guided_stable_diffuser.py:434, step_size 0.1); the product is rounded to fp32 before
 * the subtraction, like the two torch ops.  out may be latents itself (in place); a partial overlap is rejected. */
int dh_latent_step(const float* latents, const float* grad, float step_size, float* out, size_t n, void* stream);
/* Coefficients of one DDIM update, computed by the caller in fp32 exactly as diffusers 0.23 DDIMScheduler.step does on
 * 0-d fp32 tensors (alphas_cumprod[t] ** 0.5, (1 - alphas_cumprod[t]) ** 0.5, the same for the previous timestep;
 * final_alpha_cumprod when that is < 0).  divide_by_reciprocal != 0: x0 = (..) * (1.0f / sqrt_alpha_t), which is what
 * torch's CUDA division by a host scalar computes; 0: IEEE division (torch on the CPU). */
typedef struct dh_ddim_coeffs {
    float guidance_scale;        /* 7.5 (guided_stable_diffuser.py:471) */
    float sqrt_beta_t;
    float sqrt_alpha_t;
    float sqrt_alpha_prev;
    float sqrt_beta_prev;
    int32_t divide_by_reciprocal;
} dh_ddim_coeffs;
/* Classifier-free-guidance combine + DDIM update (epsilon prediction, eta = 0, no clipping / thresholding) in one pass:
 *   eps = noise_uncond + guidance_scale * (noise_text - noise_uncond)          guided_stable_diffuser.py:470-471 (and :262-263)
 *   x0  = (sample - sqrt_beta_t * eps) / sqrt_alpha_t
 *   out = sqrt_alpha_prev * x0 + sqrt_beta_prev * eps                          guided_stable_diffuser.py:474 (and :267)
 * every product / sum rounded to fp32 separately (no FMA).  noise_text == NULL: eps = noise_uncond (plain DDIM update).
 * eps_out (may be NULL) receives eps.  out may be sample itself. */
int dh_cfg_ddim_step(const float* noise_uncond, const float* noise_text, const float* sample,
                     const dh_ddim_coeffs* coeffs_host, float* out, float* eps_out, size_t n, void* stream);

/* ---- row 11 / 8(f) rank 2: hard z-buffer triangle rasteriser (mesh mode), depth_transform.py:91-195 via ------------
 * pytorch3d_renderer.py:541-941.  Semantics of pytorch3d's rasterize_meshes for faces_per_pixel = 1 (PARITY UNPINNED:
 * pytorch3d is not available).  verts (V,3) fp32 world space; faces (F,3) int32; view = X R + T; NDC = (sx X/Z, sy Y/Z).
 * Outputs per pixel: pix_to_face int32 (-1 = empty), zbuf, bary (H,W,3) (clipped, perspective corrected; -1 = empty). */
size_t dh_raster_workspace_bytes(int V, int H, int W);
int dh_rasterize_meshes(const float* verts, int V, const int32_t* faces, int F, int H, int W,
                        const float* R_host9, const float* T_host3, float sx, float sy, float blur_radius,
                        int cull_backfaces, int perspective_correct, int clip_barycentric,
                        int32_t* pix_to_face, float* zbuf, float* bary, void* ws, size_t ws_bytes, void* stream);
/* out (H,W,D+1) = hard blend of the barycentrically interpolated vertex attribute attr (V,D), alpha last, background 0 */
int dh_interpolate_face_attributes(const float* attr, int D, const int32_t* faces, const int32_t* pix_to_face,
                                   const float* bary, int H, int W, float* out, void* stream);

/* ---- mesh mode for B transforms of one scene ------------------------------------------------------
 * The geometry of B mesh-mode edits in one call: the foreground mesh (fg_verts (V_fg,3) world, fg_colors (V_fg,3) = source
 * x/(W-1), y/(H-1), flag; fg_faces (F_fg,3) fg-local ids) is moved by transform b (angle in degrees, axes_host[3b..3b+2],
 * translations_host[3b..3b+2]; bit-identical to dh_transform_points) and rendered over the background mesh (bg_verts (V_bg,3),
 * bg_faces (F_bg,3), colour flag 0) exactly as dh_rasterize_meshes renders the joined mesh [bg, fg] (fg face f = F_bg + f):
 * the background is rasterised once for all edits.  Outputs per edit b:
 *   target_z (B,H,W)  world z of the visible surface (0 = empty pixel), as the interpolated world position;
 *   corr (B,H*W,4) int64, 32-byte aligned: rows [x_src, y_src, x_dst, y_dst] in target raster order, one per pixel whose
 *                     winning face carries an interpolated flag > 0.5, source = round-half-even(carried * (W-1, H-1));
 *   n_corr[b]         device int32, rows of edit b;
 *   pix_to_face       optional (B,H,W) int32, joined face index or -1.
 * V_fg = 0 or F_fg = 0 is valid (no correspondences).  No allocation, no synchronisation; every check runs before any CUDA call:
 * DH_ERR_INVALID_ARGUMENT for NULL required pointers, B < 1, V_bg < 1, negative counts, F_fg > 0 without vertices,
 * blur_radius < 0; DH_ERR_UNSUPPORTED for B > 65535, H*W > 2^29, B*V_fg or F_bg + F_fg above 2^31 - 1.  The workspace query
 * returns 0 for sizes the call rejects. */
size_t dh_edit_mesh_batch_workspace_bytes(int B, int V_bg, int V_fg, int H, int W);
int dh_edit_mesh_batch(const float* bg_verts, int V_bg, const int32_t* bg_faces, int F_bg,
                       const float* fg_verts, const float* fg_colors, int V_fg, const int32_t* fg_faces, int F_fg,
                       int B, const float* angles_deg_host, const float* axes_host, const float* translations_host,
                       int H, int W, const float* R_host9, const float* T_host3, float sx, float sy, float blur_radius,
                       int cull_backfaces, int perspective_correct, int clip_barycentric,
                       float* target_z, int64_t* corr, int32_t* n_corr, int32_t* pix_to_face, void* ws, size_t ws_bytes,
                       void* stream);

/* ---- mesh mode for B transforms over a table of scenes -------------------------------------------
 * dh_edit_mesh_batch for edits of several images in one call.  All scenes share H, W and the camera.  Scene s has V_bg[s]
 * background vertices and F_bg[s] faces, V_fg[s] foreground vertices (with colours) and F_fg[s] faces (the host int32 arrays
 * V_bg_host, F_bg_host, V_fg_host, F_fg_host of n_scenes entries); the device arrays hold the scenes concatenated in order: bg_verts (sum V_bg,3), bg_faces (sum F_bg,3),
 * fg_verts / fg_colors (sum V_fg,3), fg_faces (sum F_fg,3), faces with scene-local vertex ids.  Edit b moves the foreground of
 * scene scene_index_host[b] by its transform (angles_deg_host[b], axes_host[3b..], translations_host[3b..]).  Outputs as for
 * dh_edit_mesh_batch, one plane / row block per edit; pix_to_face holds the joined face index of the edit's scene.
 * Contract: edit b equals, bit for bit, dh_edit_mesh_batch on scene scene_index_host[b] with that transform.  Each scene
 * referenced by an edit is rasterised once; scenes no edit references are projected but not rasterised.  One upload of the
 * descriptor tables, no allocation, no synchronisation; every check runs before any CUDA call: DH_ERR_INVALID_ARGUMENT for NULL
 * required pointers, n_scenes < 1, B < 1, a scene index outside [0, n_scenes), V_bg < 1, negative counts, F_fg > 0 without
 * vertices, a negative or NaN blur_radius, corr not 32-byte aligned; DH_ERR_UNSUPPORTED for B or n_scenes > 65535, H*W > 2^29,
 * vertex or face totals, the moved-vertex total (sum over edits of V_fg) or a scene's F_bg + F_fg above 2^31 - 1.  The workspace
 * query returns 0 for sizes the call rejects. */
size_t dh_edit_mesh_scenes_workspace_bytes(int n_scenes, const int32_t* V_bg_host, const int32_t* F_bg_host, const int32_t* V_fg_host,
                                           const int32_t* F_fg_host, int B, const int32_t* scene_index_host, int H, int W);
int dh_edit_mesh_scenes(int n_scenes, const float* bg_verts, const int32_t* bg_faces, const int32_t* V_bg_host, const int32_t* F_bg_host,
                        const float* fg_verts, const float* fg_colors, const int32_t* fg_faces, const int32_t* V_fg_host,
                        const int32_t* F_fg_host, int B, const int32_t* scene_index_host, const float* angles_deg_host,
                        const float* axes_host, const float* translations_host, int H, int W, const float* R_host9,
                        const float* T_host3, float sx, float sy, float blur_radius, int cull_backfaces, int perspective_correct,
                        int clip_barycentric, float* target_z, int64_t* corr, int32_t* n_corr, int32_t* pix_to_face, void* ws,
                        size_t ws_bytes, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DH_B200_H */
