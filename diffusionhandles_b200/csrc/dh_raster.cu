// Hard z-buffer triangle rasteriser for the reference's mesh mode (SURVEY.md 8(a) row 11, 8(f) rank 2;
// depth_transform.py:91-195 through pytorch3d_renderer.py:541-941).
//
// The reference calls pytorch3d's MeshRasterizer (faces_per_pixel = 1, blur_radius 1e-5, perspective-correct and
// clipped barycentrics, back-face culling).  pytorch3d is not installed here and no reference test pins its output, so
// this kernel follows the published semantics of pytorch3d's rasterize_meshes (SURVEY.md Appendix B) - PARITY UNPINNED:
//   * vertices: view = X R + T, NDC x = sx X / Z, y = sy Y / Z, NDC z = view z  (+x left, +y up);
//   * pixel (row i, col j) samples NDC (x, y) = (PixToNdc(W-1-j), PixToNdc(H-1-i)), pixel centres at half integers;
//   * per pixel and face: skip if the face is behind the camera, back-facing (when culling), of ~zero area or the pixel
//     is outside the bounding box grown by sqrt(blur_radius); barycentrics -> perspective correction -> clip and
//     renormalise; pz = sum bary * z; skip pz < 0; accept if inside (unclipped barycentrics > 0) or the squared
//     distance to the triangle is below blur_radius;
//   * the winner of a pixel is the lexicographic minimum of (pz, face index): ONE 64-bit atomicMin on
//     (float bits of pz << 32 | face index) - pz >= 0, so its bit pattern is order preserving.
// One thread per face walks the pixels of the face's bounding box; a second kernel recomputes the barycentrics of the
// winning face per pixel.  All arithmetic is fp32 with explicit round-to-nearest operations (no FMA contraction), so the
// NumPy restatement in the oracle reproduces it bit for bit.
#include "dh_common.cuh"

#include <math.h>
#include <string.h>

#include <vector>

namespace dh {

constexpr float kRasterEps = 1e-8f;

struct RasterCamDev {
    float R[9];     // view = X R + T (row-vector convention, like pytorch3d)
    float T[3];
    float sx, sy;   // NDC = (sx X / Z, sy Y / Z)
};

struct RasterSettings {
    float blur_radius, blur_sqrt;
    int cull_backfaces, perspective_correct, clip_barycentric;
};

__device__ __forceinline__ float ndc_range(int S1, int S2) {
    float range = 2.0f;
    if (S1 > S2) range = __fdiv_rn(__fmul_rn((float)S1, range), (float)S2);
    return range;
}

__device__ __forceinline__ float pix_to_ndc(int i, int S1, int S2) {
    const float range = ndc_range(S1, S2);
    const float offset = __fdiv_rn(range, 2.0f);
    return __fadd_rn(-offset, __fdiv_rn(__fadd_rn(__fmul_rn(range, (float)i), offset), (float)S1));
}

__device__ __forceinline__ float edge_fn(float px, float py, float ax, float ay, float bx, float by) {
    return __fsub_rn(__fmul_rn(__fsub_rn(px, ax), __fsub_rn(by, ay)), __fmul_rn(__fsub_rn(py, ay), __fsub_rn(bx, ax)));
}

__device__ __forceinline__ float seg_dist2(float px, float py, float ax, float ay, float bx, float by) {
    const float bax = __fsub_rn(bx, ax), bay = __fsub_rn(by, ay);
    const float l2 = __fadd_rn(__fmul_rn(bax, bax), __fmul_rn(bay, bay));
    if (l2 <= kRasterEps) {
        const float dx = __fsub_rn(px, bx), dy = __fsub_rn(py, by);
        return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    }
    float t = __fdiv_rn(__fadd_rn(__fmul_rn(bax, __fsub_rn(px, ax)), __fmul_rn(bay, __fsub_rn(py, ay))), l2);
    t = fminf(fmaxf(t, 0.0f), 1.0f);
    const float qx = __fadd_rn(ax, __fmul_rn(t, bax)), qy = __fadd_rn(ay, __fmul_rn(t, bay));
    const float dx = __fsub_rn(px, qx), dy = __fsub_rn(py, qy);
    return __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
}

struct Tri {
    float x0, y0, z0, x1, y1, z1, x2, y2, z2;
};

// pytorch3d CheckPixelInsideFace for one (pixel, face).  Returns true when the face covers the pixel; pz and the clipped,
// perspective-corrected barycentrics are written.
__device__ __forceinline__ bool pixel_in_face(const Tri& t, float px, float py, const RasterSettings& st, float& pz, float& b0,
                                              float& b1, float& b2) {
    const float zmax = fmaxf(t.z0, fmaxf(t.z1, t.z2));
    const float xmin = fminf(t.x0, fminf(t.x1, t.x2)) - st.blur_sqrt, xmax = fmaxf(t.x0, fmaxf(t.x1, t.x2)) + st.blur_sqrt;
    const float ymin = fminf(t.y0, fminf(t.y1, t.y2)) - st.blur_sqrt, ymax = fmaxf(t.y0, fmaxf(t.y1, t.y2)) + st.blur_sqrt;
    const bool outside = px > xmax || px < xmin || py > ymax || py < ymin;
    const float area = edge_fn(t.x0, t.y0, t.x1, t.y1, t.x2, t.y2);
    const bool back = area < 0.0f;
    const bool zero_area = area <= kRasterEps && area >= -kRasterEps;
    if (zmax < 0.0f || (st.cull_backfaces && back) || outside || zero_area) return false;
    // barycentric coordinates
    const float a = __fadd_rn(edge_fn(t.x2, t.y2, t.x0, t.y0, t.x1, t.y1), kRasterEps);
    float w0 = __fdiv_rn(edge_fn(px, py, t.x1, t.y1, t.x2, t.y2), a);
    float w1 = __fdiv_rn(edge_fn(px, py, t.x2, t.y2, t.x0, t.y0), a);
    float w2 = __fdiv_rn(edge_fn(px, py, t.x0, t.y0, t.x1, t.y1), a);
    if (st.perspective_correct) {
        const float t0 = __fmul_rn(__fmul_rn(w0, t.z1), t.z2);
        const float t1 = __fmul_rn(__fmul_rn(t.z0, w1), t.z2);
        const float t2 = __fmul_rn(__fmul_rn(t.z0, t.z1), w2);
        const float den = fmaxf(__fadd_rn(__fadd_rn(t0, t1), t2), kRasterEps);
        w0 = __fdiv_rn(t0, den); w1 = __fdiv_rn(t1, den); w2 = __fdiv_rn(t2, den);
    }
    float c0 = w0, c1 = w1, c2 = w2;
    if (st.clip_barycentric) {
        c0 = fmaxf(0.0f, fminf(1.0f, w0)); c1 = fmaxf(0.0f, fminf(1.0f, w1)); c2 = fmaxf(0.0f, fminf(1.0f, w2));
        const float s = fmaxf(__fadd_rn(__fadd_rn(c0, c1), c2), 1e-5f);
        c0 = __fdiv_rn(c0, s); c1 = __fdiv_rn(c1, s); c2 = __fdiv_rn(c2, s);
    }
    pz = __fadd_rn(__fadd_rn(__fmul_rn(c0, t.z0), __fmul_rn(c1, t.z1)), __fmul_rn(c2, t.z2));
    if (pz < 0.0f) return false;
    const bool inside = w0 > 0.0f && w1 > 0.0f && w2 > 0.0f;
    if (!inside) {
        const float d = fminf(seg_dist2(px, py, t.x0, t.y0, t.x1, t.y1),
                              fminf(seg_dist2(px, py, t.x0, t.y0, t.x2, t.y2), seg_dist2(px, py, t.x1, t.y1, t.x2, t.y2)));
        if (d >= st.blur_radius) return false;
    }
    b0 = c0; b1 = c1; b2 = c2;
    return true;
}

__global__ void __launch_bounds__(256) raster_project_kernel(const float* __restrict__ verts, int V, RasterCamDev cam,
                                                             float* __restrict__ ndc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= V) return;
    const float X = verts[3 * (size_t)i], Y = verts[3 * (size_t)i + 1], Z = verts[3 * (size_t)i + 2];
    // view = X R + T, left-to-right fp32 accumulation (identity R / zero T for every reference caller -> exact)
    float v[3];
#pragma unroll
    for (int c = 0; c < 3; ++c)
        v[c] = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(X, cam.R[c]), __fmul_rn(Y, cam.R[3 + c])), __fmul_rn(Z, cam.R[6 + c])), cam.T[c]);
    // homogeneous divide with pytorch3d's eps clamp on the denominator
    float den = v[2];
    const float ad = fmaxf(fabsf(den), 1e-8f);      // (MeshRasterizer passes eps = None -> no clamp; kept tiny for z = 0)
    den = den < 0.0f ? -ad : ad;
    ndc[3 * (size_t)i] = __fdiv_rn(__fmul_rn(cam.sx, v[0]), den);
    ndc[3 * (size_t)i + 1] = __fdiv_rn(__fmul_rn(cam.sy, v[1]), den);
    ndc[3 * (size_t)i + 2] = v[2];
}

__device__ __forceinline__ Tri load_tri(const float* __restrict__ ndc, const int32_t* __restrict__ faces, int f) {
    const int i0 = faces[3 * (size_t)f], i1 = faces[3 * (size_t)f + 1], i2 = faces[3 * (size_t)f + 2];
    Tri t;
    t.x0 = ndc[3 * (size_t)i0]; t.y0 = ndc[3 * (size_t)i0 + 1]; t.z0 = ndc[3 * (size_t)i0 + 2];
    t.x1 = ndc[3 * (size_t)i1]; t.y1 = ndc[3 * (size_t)i1 + 1]; t.z1 = ndc[3 * (size_t)i1 + 2];
    t.x2 = ndc[3 * (size_t)i2]; t.y2 = ndc[3 * (size_t)i2 + 1]; t.z2 = ndc[3 * (size_t)i2 + 2];
    return t;
}

// component d of a (V,D) vertex attribute interpolated with the barycentrics of face (i0, i1, i2)
__device__ __forceinline__ float interp_attr(const float* __restrict__ attr, int D, int d, int i0, int i1, int i2, float b0, float b1,
                                             float b2) {
    return __fadd_rn(__fadd_rn(__fmul_rn(attr[(size_t)i0 * D + d], b0), __fmul_rn(attr[(size_t)i1 * D + d], b1)),
                     __fmul_rn(attr[(size_t)i2 * D + d], b2));
}

// one face: walk the pixels of its bounding box and offer (pz, key_face) to the z-buffer of every pixel it covers
__device__ __forceinline__ void raster_face(const Tri& t, unsigned int key_face, int H, int W, const RasterSettings& st,
                                            unsigned long long* keys) {
    const float zmax = fmaxf(t.z0, fmaxf(t.z1, t.z2));
    if (zmax < 0.0f) return;
    // candidate pixel range from the blur-grown bounding box (conservative; the exact test is repeated per pixel)
    const float xmin = fminf(t.x0, fminf(t.x1, t.x2)) - st.blur_sqrt, xmax = fmaxf(t.x0, fmaxf(t.x1, t.x2)) + st.blur_sqrt;
    const float ymin = fminf(t.y0, fminf(t.y1, t.y2)) - st.blur_sqrt, ymax = fmaxf(t.y0, fmaxf(t.y1, t.y2)) + st.blur_sqrt;
    if (!(xmin == xmin) || !(xmax == xmax) || !(ymin == ymin) || !(ymax == ymax)) return;     // NaN vertices
    const float rx = ndc_range(W, H), ry = ndc_range(H, W);
    // ndc = -r/2 + (r i + r/2) / S   <=>   i = ((ndc + r/2) S - r/2) / r
    auto to_idx = [](float v, float r, int S) { return ((v + 0.5f * r) * (float)S - 0.5f * r) / r; };
    int xi0 = (int)floorf(fminf(fmaxf(to_idx(xmin, rx, W), -2.0f), (float)W + 1.0f)) - 1;
    int xi1 = (int)ceilf(fminf(fmaxf(to_idx(xmax, rx, W), -2.0f), (float)W + 1.0f)) + 1;
    int yi0 = (int)floorf(fminf(fmaxf(to_idx(ymin, ry, H), -2.0f), (float)H + 1.0f)) - 1;
    int yi1 = (int)ceilf(fminf(fmaxf(to_idx(ymax, ry, H), -2.0f), (float)H + 1.0f)) + 1;
    xi0 = max(xi0, 0); yi0 = max(yi0, 0); xi1 = min(xi1, W - 1); yi1 = min(yi1, H - 1);
    for (int yidx = yi0; yidx <= yi1; ++yidx) {
        const float py = pix_to_ndc(yidx, H, W);
        for (int xidx = xi0; xidx <= xi1; ++xidx) {
            const float px = pix_to_ndc(xidx, W, H);
            float pz, b0, b1, b2;
            if (!pixel_in_face(t, px, py, st, pz, b0, b1, b2)) continue;
            // image row / column: both axes are reversed (+x left, +y up)
            const int row = H - 1 - yidx, col = W - 1 - xidx;
            const unsigned long long key = ((unsigned long long)__float_as_uint(pz) << 32) | key_face;
            unsigned long long* k = keys + (size_t)row * W + col;
            if (key < *(volatile unsigned long long*)k) atomicMin(k, key);
        }
    }
}

__global__ void __launch_bounds__(128) raster_faces_kernel(const float* __restrict__ ndc, const int32_t* __restrict__ faces, int F,
                                                           int H, int W, RasterSettings st, unsigned long long* keys) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    raster_face(load_tri(ndc, faces, f), (unsigned int)f, H, W, st, keys);
}

__global__ void __launch_bounds__(256) raster_resolve_kernel(const float* __restrict__ ndc, const int32_t* __restrict__ faces, int H,
                                                             int W, RasterSettings st, const unsigned long long* __restrict__ keys,
                                                             int32_t* __restrict__ pix_to_face, float* __restrict__ zbuf,
                                                             float* __restrict__ bary) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= H * W) return;
    const unsigned long long key = keys[q];
    int f = -1;
    float pz = -1.0f, b0 = -1.0f, b1 = -1.0f, b2 = -1.0f;       // pytorch3d fills empty pixels with -1
    if (key != 0xFFFFFFFFFFFFFFFFull) {
        f = (int)(key & 0xFFFFFFFFull);
        const int row = q / W, col = q - row * W;
        const float px = pix_to_ndc(W - 1 - col, W, H), py = pix_to_ndc(H - 1 - row, H, W);
        const Tri t = load_tri(ndc, faces, f);
        pixel_in_face(t, px, py, st, pz, b0, b1, b2);
    }
    pix_to_face[q] = f;
    zbuf[q] = pz;
    bary[3 * (size_t)q] = b0; bary[3 * (size_t)q + 1] = b1; bary[3 * (size_t)q + 2] = b2;
}

// hard blend of a barycentrically interpolated vertex attribute: out (H,W,D+1), alpha in the last channel,
// background 0 (pytorch3d_renderer.py:56-142, :487-537)
__global__ void __launch_bounds__(256) raster_interpolate_kernel(const float* __restrict__ attr, int D, const int32_t* __restrict__ faces,
                                                                 const int32_t* __restrict__ pix_to_face, const float* __restrict__ bary,
                                                                 int P, float* __restrict__ out) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= P) return;
    const int f = pix_to_face[q];
    float* o = out + (size_t)q * (D + 1);
    if (f < 0) {
        for (int d = 0; d <= D; ++d) o[d] = 0.0f;
        return;
    }
    const int i0 = faces[3 * (size_t)f], i1 = faces[3 * (size_t)f + 1], i2 = faces[3 * (size_t)f + 2];
    const float b0 = bary[3 * (size_t)q], b1 = bary[3 * (size_t)q + 1], b2 = bary[3 * (size_t)q + 2];
    for (int d = 0; d < D; ++d) o[d] = interp_attr(attr, D, d, i0, i1, i2, b0, b1, b2);
    o[D] = 1.0f;
}

static size_t raster_layout(int V, int P, size_t* o_ndc, size_t* o_keys) {
    size_t o = 0;
    *o_ndc = o;  o = align_up(o + sizeof(float) * 3 * (size_t)V, 256);
    *o_keys = o; o = align_up(o + sizeof(unsigned long long) * (size_t)P, 256);
    return o;
}


// ------------------------------------------------------------------------------------------------
// Mesh mode for B rigid transforms of one scene's foreground (dh_edit_mesh_batch).
//
// A pixel's z-buffer entry is the minimum of (pz bits << 32 | face index) over the faces that cover it, and a minimum does not
// depend on how the faces are split: the minimum over bg u fg is the minimum of the bg minimum and the fg minimum.  So the
// background faces are rasterised ONCE, their keys are copied to every edit, and each edit's moved foreground faces go on top
// with the index they have in the joined mesh (F_bg + f).  The result is bit-identical to rasterising [bg, fg] joined, and the
// background faces still win exact ties.  Each (pixel, edit) winner is then resolved straight to what mesh mode reads off the
// render - the world z and, for a foreground winner, the carried source pixel - without barycentric or attribute buffers.
// ------------------------------------------------------------------------------------------------
constexpr int kMeshTile = 1024;                 // pixels per compaction tile
constexpr int kMeshTileThreads = kMeshTile / 4; // 4 consecutive pixels per thread (raster order = thread order)
constexpr int kMaxGridY = 65535;

struct MeshBatchScene {
    const float* bg_ndc;      // (V_bg,3)
    const float* bg_verts;    // (V_bg,3) world
    const int32_t* bg_faces;  // (F_bg,3)
    int F_bg;
    const float* fg_ndc;      // (B,V_fg,3)
    const float* fg_world;    // (B,V_fg,3) transformed world vertices
    const float* fg_colors;   // (V_fg,3) source x/(W-1), y/(H-1), flag
    const int32_t* fg_faces;  // (F_fg,3) fg-local vertex ids
    int V_fg;
};

// keys of the background raster (edit 0) -> every other edit
__global__ void __launch_bounds__(256) raster_keys_broadcast_kernel(unsigned long long* keys, int P, int B) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= P) return;
    const unsigned long long k = keys[q];
    for (int b = 1; b < B; ++b) keys[(size_t)b * P + q] = k;
}

// the foreground faces of every edit (blockIdx.y = edit), keyed with their index in the joined mesh
__global__ void __launch_bounds__(128) raster_faces_batch_kernel(const float* __restrict__ ndc, int V, const int32_t* __restrict__ faces,
                                                                 int F, int key_base, int H, int W, RasterSettings st,
                                                                 unsigned long long* keys) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    const int b = blockIdx.y;
    raster_face(load_tri(ndc + 3 * (size_t)V * b, faces, f), (unsigned int)(key_base + f), H, W, st, keys + (size_t)b * H * W);
}

// Pixel q of edit b with z-buffer entry `key`: returns the world z of the winning surface (world_position[..., 2]: 0 when the pixel
// is empty).  `emit` is set when a foreground face wins and its interpolated flag exceeds 0.5, with the source pixel it carries,
// rounded half-to-even like torch.round.  A background face carries the colour (x, y, 0): its flag is exactly 0, it never emits.
__device__ __forceinline__ float mesh_resolve(const MeshBatchScene& s, int b, int q, unsigned long long key, int H, int W,
                                              const RasterSettings& st, bool& emit, float& src_x, float& src_y) {
    emit = false;
    if (key == 0xFFFFFFFFFFFFFFFFull) return 0.0f;
    const int f = (int)(key & 0xFFFFFFFFull);
    const bool fg = f >= s.F_bg;
    const int lf = fg ? f - s.F_bg : f;
    const float* ndc = fg ? s.fg_ndc + 3 * (size_t)s.V_fg * b : s.bg_ndc;
    const float* verts = fg ? s.fg_world + 3 * (size_t)s.V_fg * b : s.bg_verts;
    const int32_t* faces = fg ? s.fg_faces : s.bg_faces;
    const int row = q / W, col = q - row * W;
    const float px = pix_to_ndc(W - 1 - col, W, H), py = pix_to_ndc(H - 1 - row, H, W);
    float pz, b0 = -1.0f, b1 = -1.0f, b2 = -1.0f;
    pixel_in_face(load_tri(ndc, faces, lf), px, py, st, pz, b0, b1, b2);
    const int i0 = faces[3 * (size_t)lf], i1 = faces[3 * (size_t)lf + 1], i2 = faces[3 * (size_t)lf + 2];
    const float z = interp_attr(verts, 3, 2, i0, i1, i2, b0, b1, b2);
    if (fg && interp_attr(s.fg_colors, 3, 2, i0, i1, i2, b0, b1, b2) > 0.5f) {
        emit = true;
        src_x = rintf(__fmul_rn(interp_attr(s.fg_colors, 3, 0, i0, i1, i2, b0, b1, b2), (float)(W - 1)));
        src_y = rintf(__fmul_rn(interp_attr(s.fg_colors, 3, 1, i0, i1, i2, b0, b1, b2), (float)(H - 1)));
    }
    return z;
}

// pass 1 over (pixel, edit): target z (+ pix_to_face when asked for) and the number of correspondences per tile
__global__ void __launch_bounds__(kMeshTileThreads) mesh_resolve_count_kernel(MeshBatchScene s, const unsigned long long* __restrict__ keys,
                                                                               int H, int W, int ntiles, RasterSettings st,
                                                                               float* __restrict__ target_z, int32_t* __restrict__ pix_to_face,
                                                                               int32_t* __restrict__ tile_counts) {
    __shared__ int warp_sums[32];
    const int b = blockIdx.y, tile = blockIdx.x, P = H * W;
    const size_t eo = (size_t)b * P;
    const int q0 = tile * kMeshTile + threadIdx.x * 4;
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + i;
        if (q >= P) continue;
        const unsigned long long key = keys[eo + q];
        bool emit;
        float sx, sy;
        target_z[eo + q] = mesh_resolve(s, b, q, key, H, W, st, emit, sx, sy);
        c += emit;
        if (pix_to_face) pix_to_face[eo + q] = key == 0xFFFFFFFFFFFFFFFFull ? -1 : (int32_t)(key & 0xFFFFFFFFull);
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if (lane_id() == 0) warp_sums[warp_id()] = c;
    __syncthreads();
    if (warp_id() == 0) {
        int t = lane_id() < (int)(blockDim.x >> 5) ? warp_sums[lane_id()] : 0;
        t = __reduce_add_sync(0xFFFFFFFFu, t);
        if (lane_id() == 0) tile_counts[b * ntiles + tile] = t;
    }
}

// pass 2: the rows [x_src, y_src, x_dst, y_dst] of every edit in target raster order (tile offsets from the counts, then a block
// scan); only foreground winners are resolved again.  The last tile of an edit publishes n_corr.
__global__ void __launch_bounds__(kMeshTileThreads) mesh_emit_kernel(MeshBatchScene s, const unsigned long long* __restrict__ keys,
                                                                      int H, int W, int ntiles, RasterSettings st,
                                                                      const int32_t* __restrict__ tile_counts, int64_t* __restrict__ corr,
                                                                      int32_t* __restrict__ n_corr) {
    __shared__ int scan_smem[33];
    __shared__ int base_smem;
    const int b = blockIdx.y, tile = blockIdx.x, P = H * W;
    if (tile_counts[b * ntiles + tile] == 0 && tile != ntiles - 1) return;     // nothing to emit (uniform over the block)
    int part = 0;
    for (int t = threadIdx.x; t < tile; t += blockDim.x) part += tile_counts[b * ntiles + t];
    int tot;
    block_exclusive_scan(part, scan_smem, tot);
    if (threadIdx.x == 0) base_smem = tot;
    __syncthreads();
    const int base = base_smem;
    const size_t eo = (size_t)b * P;
    const int q0 = tile * kMeshTile + threadIdx.x * 4;
    unsigned kmask = 0;
    float sx[4], sy[4];          // rounded source coordinates, converted to int64 at the store
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + i;
        sx[i] = sy[i] = 0.0f;
        if (q >= P) continue;
        const unsigned long long key = keys[eo + q];
        if (key == 0xFFFFFFFFFFFFFFFFull || (int)(key & 0xFFFFFFFFull) < s.F_bg) continue;
        bool emit;
        mesh_resolve(s, b, q, key, H, W, st, emit, sx[i], sy[i]);
        kmask |= (unsigned)emit << i;
    }
    int total;
    int pos = base + block_exclusive_scan(__popc(kmask), scan_smem, total);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!((kmask >> i) & 1u)) continue;
        const int q = q0 + i, row = q / W;
        longlong4 v;
        v.x = (long long)sx[i]; v.y = (long long)sy[i]; v.z = q - row * W; v.w = row;
        *reinterpret_cast<longlong4*>(corr + (eo + pos) * 4) = v;
        ++pos;
    }
    if (tile == ntiles - 1 && threadIdx.x == 0) n_corr[b] = base + total;
}

struct MeshBatchLayout {
    size_t partial, edits, bg_ndc, fg_world, fg_ndc, keys, tile_counts, total;
};

static MeshBatchLayout mesh_batch_layout(int B, int V_bg, int V_fg, int H, int W) {
    const size_t P = (size_t)H * W, ntiles = (P + kMeshTile - 1) / kMeshTile;
    MeshBatchLayout L;
    size_t o = 0;
    L.partial = o;     o = align_up(o + sizeof(double) * 3 * kTpMaxPartials, 256);
    L.edits = o;       o = align_up(o + sizeof(TpEdit) * (size_t)B, 256);
    L.bg_ndc = o;      o = align_up(o + sizeof(float) * 3 * (size_t)V_bg, 256);
    L.fg_world = o;    o = align_up(o + sizeof(float) * 3 * (size_t)V_fg * B, 256);
    L.fg_ndc = o;      o = align_up(o + sizeof(float) * 3 * (size_t)V_fg * B, 256);
    L.keys = o;        o = align_up(o + sizeof(unsigned long long) * P * B, 256);
    L.tile_counts = o; o = align_up(o + sizeof(int32_t) * ntiles * B, 256);
    L.total = o;
    return L;
}

static RasterCamDev make_raster_cam(const float* R_host9, const float* T_host3, float sx, float sy) {
    RasterCamDev cam;
    memcpy(cam.R, R_host9, sizeof(cam.R));
    memcpy(cam.T, T_host3, sizeof(cam.T));
    cam.sx = sx; cam.sy = sy;
    return cam;
}

static RasterSettings make_raster_settings(float blur_radius, int cull_backfaces, int perspective_correct, int clip_barycentric) {
    RasterSettings st;
    st.blur_radius = blur_radius; st.blur_sqrt = sqrtf(blur_radius);
    st.cull_backfaces = cull_backfaces; st.perspective_correct = perspective_correct; st.clip_barycentric = clip_barycentric;
    return st;
}

// size checks shared by the call and its workspace query
static int mesh_batch_sizes(int B, int V_bg, int F_bg, int V_fg, int F_fg, int H, int W) {
    if (B < 1 || V_bg < 1 || F_bg < 0 || V_fg < 0 || F_fg < 0 || H < 1 || W < 1) return DH_ERR_INVALID_ARGUMENT;
    if (F_fg > 0 && V_fg == 0) return DH_ERR_INVALID_ARGUMENT;       // faces without vertices
    if (B > kMaxGridY) return DH_ERR_UNSUPPORTED;                     // one grid row per edit
    if ((long long)H * W > (1ll << 29)) return DH_ERR_UNSUPPORTED;
    if ((long long)B * V_fg > 0x7FFFFFFFll) return DH_ERR_UNSUPPORTED; // the moved vertices are projected as one flat array
    if ((long long)F_bg + F_fg > 0x7FFFFFFFll) return DH_ERR_UNSUPPORTED; // joined face indices are 31-bit in the keys
    return DH_OK;
}

// ------------------------------------------------------------------------------------------------
// Mesh mode for B rigid transforms over a table of scenes (dh_edit_mesh_scenes): the one-scene scheme above per scene.  Each
// scene's background faces are rasterised ONCE, into the key plane of the first edit of that scene, their keys are copied to the
// scene's other edits, and each edit's moved foreground faces go on top with the index they have in the joined mesh of its scene
// (F_bg + f).  Edit b is bit-identical to dh_edit_mesh_batch on its scene.
//
// dh_edit_mesh_batch keeps its own kernels: run through this path its device time was about 1 % longer at B = 1..16 (DESIGN.md 5),
// from the per-block descriptor reads of the foreground raster, the moved-vertex transform and the emit pass.
//
// Per-scene and per-edit offsets live in two small device tables (SceneDesc, SceneEdit; one upload).  Grids whose x extent
// depends on a scene (face blocks, centroid blocks, moved vertices) are sized by the largest one and the blocks past a smaller
// scene's end exit at once: no search over per-edit face ranges is needed, and an idle block costs a block launch.
// ------------------------------------------------------------------------------------------------
constexpr unsigned long long kNoKey = 0xFFFFFFFFFFFFFFFFull;

// the concatenated arrays of a scene batch and its device tables
struct MeshScenes {
    const float* bg_ndc;      // (sum V_bg,3)
    const float* bg_verts;    // (sum V_bg,3) world
    const int32_t* bg_faces;  // (sum F_bg,3) scene-local
    const float* fg_ndc;      // (sum over edits of V_fg,3)
    const float* fg_world;    // (sum over edits of V_fg,3) transformed world vertices
    const float* fg_colors;   // (sum V_fg,3) source x/(W-1), y/(H-1), flag
    const int32_t* fg_faces;  // (sum F_fg,3) scene-local
    const SceneDesc* scenes;
    const SceneEdit* edits;
};

// the arrays of edit b's scene, as mesh_resolve reads them
struct MeshEditScene {
    const float* bg_ndc;
    const float* bg_verts;
    const int32_t* bg_faces;
    int F_bg;
    const float* fg_ndc;      // (V_fg,3) of this edit
    const float* fg_world;    // (V_fg,3) of this edit
    const float* fg_colors;
    const int32_t* fg_faces;
};

__device__ __forceinline__ MeshEditScene mesh_edit_scene(const MeshScenes& m, int b) {
    const SceneEdit& e = m.edits[b];
    const int out0 = e.out0;
    const SceneDesc& sc = m.scenes[e.scene];
    MeshEditScene s;
    s.bg_ndc = m.bg_ndc + 3 * (size_t)sc.bg_v0;
    s.bg_verts = m.bg_verts + 3 * (size_t)sc.bg_v0;
    s.bg_faces = m.bg_faces + 3 * (size_t)sc.bg_f0;
    s.F_bg = sc.F_bg;
    s.fg_ndc = m.fg_ndc + 3 * (size_t)out0;
    s.fg_world = m.fg_world + 3 * (size_t)out0;
    s.fg_colors = m.fg_colors + 3 * (size_t)sc.fg_v0;
    s.fg_faces = m.fg_faces + 3 * (size_t)sc.fg_f0;
    return s;
}

// the key plane (KS keys, KS even, 16-byte aligned) of every used scene's background raster <- empty
__global__ void __launch_bounds__(256) raster_keys_clear_kernel(const SceneDesc* __restrict__ scenes, int KS, unsigned long long* keys) {
    const int plane = scenes[blockIdx.y].plane;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (plane < 0 || 2 * i >= KS) return;
    reinterpret_cast<ulonglong2*>(keys + (size_t)plane * KS)[i] = make_ulonglong2(kNoKey, kNoKey);
}

// the background faces of every used scene (blockIdx.y = scene) into that scene's key plane
__global__ void raster_faces_scenes_kernel(const float* __restrict__ ndc, const int32_t* __restrict__ faces,
                                                                  const SceneDesc* __restrict__ scenes, int H, int W, int KS,
                                                                  RasterSettings st, unsigned long long* keys) {
    const SceneDesc* sc = scenes + blockIdx.y;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    const int plane = sc->plane;
    if (plane < 0 || f >= sc->F_bg) return;
    const Tri t = load_tri(ndc + 3 * (size_t)sc->bg_v0, faces + 3 * (size_t)sc->bg_f0, f);
    raster_face(t, (unsigned int)f, H, W, st, keys + (size_t)plane * KS);
}

// keys of edit b (blockIdx.y) <- the background raster of its scene, 16 bytes per thread; the edit holding the raster is skipped
__global__ void __launch_bounds__(256) raster_keys_scenes_broadcast_kernel(const SceneDesc* __restrict__ scenes, const SceneEdit* __restrict__ edits,
                                                                    int KS, unsigned long long* keys) {
    const int b = blockIdx.y;
    const int src = scenes[edits[b].scene].plane;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (src == b || 2 * i >= KS) return;
    reinterpret_cast<ulonglong2*>(keys + (size_t)b * KS)[i] = reinterpret_cast<const ulonglong2*>(keys + (size_t)src * KS)[i];
}

// the moved foreground faces of every edit (blockIdx.y = edit), keyed with their index in the joined mesh of its scene
__global__ void raster_faces_edits_kernel(const float* __restrict__ ndc, const int32_t* __restrict__ faces,
                                                                 const SceneDesc* __restrict__ scenes, const SceneEdit* __restrict__ edits,
                                                                 int H, int W, int KS, RasterSettings st, unsigned long long* keys) {
    const int b = blockIdx.y;
    const SceneDesc* sc = scenes + edits[b].scene;
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= sc->F_fg) return;
    const Tri t = load_tri(ndc + 3 * (size_t)edits[b].out0, faces + 3 * (size_t)sc->fg_f0, f);
    raster_face(t, (unsigned int)(sc->F_bg + f), H, W, st, keys + (size_t)b * KS);
}

// Pixel q with z-buffer entry `key` in an edit of scene s: returns the world z of the winning surface (world_position[..., 2]: 0
// when the pixel is empty).  `emit` is set when a foreground face wins and its interpolated flag exceeds 0.5, with the source pixel
// it carries, rounded half-to-even like torch.round.  A background face carries the colour (x, y, 0): its flag is exactly 0, it
// never emits.
__device__ __forceinline__ float mesh_scenes_resolve(const MeshEditScene& s, int q, unsigned long long key, int H, int W, const RasterSettings& st,
                                              bool& emit, float& src_x, float& src_y) {
    emit = false;
    if (key == kNoKey) return 0.0f;
    const int f = (int)(key & 0xFFFFFFFFull);
    const bool fg = f >= s.F_bg;
    const int lf = fg ? f - s.F_bg : f;
    const float* ndc = fg ? s.fg_ndc : s.bg_ndc;
    const float* verts = fg ? s.fg_world : s.bg_verts;
    const int32_t* faces = fg ? s.fg_faces : s.bg_faces;
    const int row = q / W, col = q - row * W;
    const float px = pix_to_ndc(W - 1 - col, W, H), py = pix_to_ndc(H - 1 - row, H, W);
    float pz, b0 = -1.0f, b1 = -1.0f, b2 = -1.0f;
    pixel_in_face(load_tri(ndc, faces, lf), px, py, st, pz, b0, b1, b2);
    const int i0 = faces[3 * (size_t)lf], i1 = faces[3 * (size_t)lf + 1], i2 = faces[3 * (size_t)lf + 2];
    const float z = interp_attr(verts, 3, 2, i0, i1, i2, b0, b1, b2);
    if (fg && interp_attr(s.fg_colors, 3, 2, i0, i1, i2, b0, b1, b2) > 0.5f) {
        emit = true;
        src_x = rintf(__fmul_rn(interp_attr(s.fg_colors, 3, 0, i0, i1, i2, b0, b1, b2), (float)(W - 1)));
        src_y = rintf(__fmul_rn(interp_attr(s.fg_colors, 3, 1, i0, i1, i2, b0, b1, b2), (float)(H - 1)));
    }
    return z;
}

// pass 1 over (pixel, edit): target z (+ pix_to_face when asked for) and the number of correspondences per tile
__global__ void __launch_bounds__(kMeshTileThreads) mesh_scenes_resolve_count_kernel(MeshScenes m, const unsigned long long* __restrict__ keys,
                                                                               int H, int W, int KS, int ntiles, RasterSettings st,
                                                                               float* __restrict__ target_z, int32_t* __restrict__ pix_to_face,
                                                                               int32_t* __restrict__ tile_counts) {
    __shared__ int warp_sums[32];
    const int b = blockIdx.y, tile = blockIdx.x, P = H * W;
    const MeshEditScene s = mesh_edit_scene(m, b);
    const size_t eo = (size_t)b * P, ko = (size_t)b * KS;
    const int q0 = tile * kMeshTile + threadIdx.x * 4;
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + i;
        if (q >= P) continue;
        const unsigned long long key = keys[ko + q];
        bool emit;
        float sx, sy;
        target_z[eo + q] = mesh_scenes_resolve(s, q, key, H, W, st, emit, sx, sy);
        c += emit;
        if (pix_to_face) pix_to_face[eo + q] = key == kNoKey ? -1 : (int32_t)(key & 0xFFFFFFFFull);
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if (lane_id() == 0) warp_sums[warp_id()] = c;
    __syncthreads();
    if (warp_id() == 0) {
        int t = lane_id() < (int)(blockDim.x >> 5) ? warp_sums[lane_id()] : 0;
        t = __reduce_add_sync(0xFFFFFFFFu, t);
        if (lane_id() == 0) tile_counts[b * ntiles + tile] = t;
    }
}

// pass 2: the rows [x_src, y_src, x_dst, y_dst] of every edit in target raster order (tile offsets from the counts, then a block
// scan); only foreground winners are resolved again.  The last tile of an edit publishes n_corr.
__global__ void __launch_bounds__(kMeshTileThreads) mesh_scenes_emit_kernel(MeshScenes m, const unsigned long long* __restrict__ keys,
                                                                      int H, int W, int KS, int ntiles, RasterSettings st,
                                                                      const int32_t* __restrict__ tile_counts, int64_t* __restrict__ corr,
                                                                      int32_t* __restrict__ n_corr) {
    __shared__ int scan_smem[33];
    __shared__ int base_smem;
    const int b = blockIdx.y, tile = blockIdx.x, P = H * W;
    if (tile_counts[b * ntiles + tile] == 0 && tile != ntiles - 1) return;     // nothing to emit (uniform over the block)
    const MeshEditScene s = mesh_edit_scene(m, b);
    int part = 0;
    for (int t = threadIdx.x; t < tile; t += blockDim.x) part += tile_counts[b * ntiles + t];
    int tot;
    block_exclusive_scan(part, scan_smem, tot);
    if (threadIdx.x == 0) base_smem = tot;
    __syncthreads();
    const int base = base_smem;
    const size_t eo = (size_t)b * P, ko = (size_t)b * KS;
    const int q0 = tile * kMeshTile + threadIdx.x * 4;
    unsigned kmask = 0;
    float sx[4], sy[4];          // rounded source coordinates, converted to int64 at the store
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int q = q0 + i;
        sx[i] = sy[i] = 0.0f;
        if (q >= P) continue;
        const unsigned long long key = keys[ko + q];
        if (key == kNoKey || (int)(key & 0xFFFFFFFFull) < s.F_bg) continue;
        bool emit;
        mesh_scenes_resolve(s, q, key, H, W, st, emit, sx[i], sy[i]);
        kmask |= (unsigned)emit << i;
    }
    int total;
    int pos = base + block_exclusive_scan(__popc(kmask), scan_smem, total);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!((kmask >> i) & 1u)) continue;
        const int q = q0 + i, row = q / W;
        longlong4 v;
        v.x = (long long)sx[i]; v.y = (long long)sy[i]; v.z = q - row * W; v.w = row;
        *reinterpret_cast<longlong4*>(corr + (eo + pos) * 4) = v;
        ++pos;
    }
    if (tile == ntiles - 1 && threadIdx.x == 0) n_corr[b] = base + total;
}

// Host view of a scene batch: the sizes every check and every launch needs, computed from the host count arrays.
struct MeshScenesPlan {
    long long V_bg, F_bg, V_fg, F_fg;   // totals over the scenes
    long long moved;                    // sum over edits of V_fg of the edit's scene
    int max_F_bg, max_F_fg, max_V_fg;   // over the scenes an edit uses (foreground: per edit)
    int tp_partials, max_tp_blocks;     // centroid partial sums over the scenes, and the most of one scene
    int KS, ntiles;                     // key plane stride (even), compaction tiles per edit
};

// every size check of dh_edit_mesh_scenes and its workspace query, before anything else
static int mesh_scenes_plan(int n_scenes, const int32_t* V_bg, const int32_t* F_bg, const int32_t* V_fg, const int32_t* F_fg, int B,
                            const int32_t* scene_index, int H, int W, MeshScenesPlan& p) {
    if (!V_bg || !F_bg || !V_fg || !F_fg || !scene_index) return DH_ERR_INVALID_ARGUMENT;
    if (n_scenes < 1 || B < 1 || H < 1 || W < 1) return DH_ERR_INVALID_ARGUMENT;
    if (n_scenes > kMaxGridY || B > kMaxGridY) return DH_ERR_UNSUPPORTED;   // one grid row per scene / per edit
    p = MeshScenesPlan{};
    bool too_big = false;
    for (int s = 0; s < n_scenes; ++s) {
        if (V_bg[s] < 1 || F_bg[s] < 0 || V_fg[s] < 0 || F_fg[s] < 0) return DH_ERR_INVALID_ARGUMENT;
        if (F_fg[s] > 0 && V_fg[s] == 0) return DH_ERR_INVALID_ARGUMENT;     // faces without vertices
        p.V_bg += V_bg[s]; p.F_bg += F_bg[s]; p.V_fg += V_fg[s]; p.F_fg += F_fg[s];
        too_big |= (long long)F_bg[s] + F_fg[s] > 0x7FFFFFFFll;               // joined face indices are 31-bit in the keys
        p.tp_partials += tp_partial_blocks(V_fg[s]);
    }
    for (int b = 0; b < B; ++b) {
        const int s = scene_index[b];
        if (s < 0 || s >= n_scenes) return DH_ERR_INVALID_ARGUMENT;
        p.moved += V_fg[s];
        p.max_F_bg = max(p.max_F_bg, F_bg[s]);
        p.max_F_fg = max(p.max_F_fg, F_fg[s]);
        p.max_V_fg = max(p.max_V_fg, V_fg[s]);
        p.max_tp_blocks = max(p.max_tp_blocks, tp_partial_blocks(V_fg[s]));
    }
    if ((long long)H * W > (1ll << 29)) return DH_ERR_UNSUPPORTED;
    // vertex and face totals are indexed with 31-bit offsets; the moved vertices are projected as one flat array
    if (too_big || p.V_bg > 0x7FFFFFFFll || p.F_bg > 0x7FFFFFFFll || p.V_fg > 0x7FFFFFFFll || p.F_fg > 0x7FFFFFFFll ||
        p.moved > 0x7FFFFFFFll)
        return DH_ERR_UNSUPPORTED;
    const int P = H * W;
    p.KS = (P + 1) & ~1;
    p.ntiles = (P + kMeshTile - 1) / kMeshTile;
    return DH_OK;
}

struct MeshScenesLayout {
    size_t scenes, edits, partial, bg_ndc, fg_world, fg_ndc, keys, tile_counts, total;
};

static MeshScenesLayout mesh_scenes_layout(int n_scenes, int B, const MeshScenesPlan& p) {
    MeshScenesLayout L;
    size_t o = 0;
    L.scenes = o;      o = align_up(o + sizeof(SceneDesc) * (size_t)n_scenes, 16);
    L.edits = o;       o = align_up(o + sizeof(SceneEdit) * (size_t)B, 256);       // [scenes, edits]: one upload
    L.partial = o;     o = align_up(o + sizeof(double) * 3 * (size_t)p.tp_partials, 256);
    L.bg_ndc = o;      o = align_up(o + sizeof(float) * 3 * (size_t)p.V_bg, 256);
    L.fg_world = o;    o = align_up(o + sizeof(float) * 3 * (size_t)p.moved, 256);
    L.fg_ndc = o;      o = align_up(o + sizeof(float) * 3 * (size_t)p.moved, 256);
    L.keys = o;        o = align_up(o + sizeof(unsigned long long) * (size_t)p.KS * B, 256);
    L.tile_counts = o; o = align_up(o + sizeof(int32_t) * (size_t)p.ntiles * B, 256);
    L.total = o;
    return L;
}

static size_t mesh_scenes_workspace(int n_scenes, const int32_t* V_bg, const int32_t* F_bg, const int32_t* V_fg, const int32_t* F_fg,
                                    int B, const int32_t* scene_index, int H, int W) {
    MeshScenesPlan p;
    if (mesh_scenes_plan(n_scenes, V_bg, F_bg, V_fg, F_fg, B, scene_index, H, W, p) != DH_OK) return 0;
    return mesh_scenes_layout(n_scenes, B, p).total;
}

static int mesh_scenes(int n_scenes, const float* bg_verts, const int32_t* bg_faces, const int32_t* V_bg, const int32_t* F_bg,
                       const float* fg_verts, const float* fg_colors, const int32_t* fg_faces, const int32_t* V_fg, const int32_t* F_fg,
                       int B, const int32_t* scene_index, const float* angles_deg_host, const float* axes_host,
                       const float* translations_host, int H, int W, const float* R_host9, const float* T_host3, float sx, float sy,
                       float blur_radius, int cull_backfaces, int perspective_correct, int clip_barycentric, float* target_z,
                       int64_t* corr, int32_t* n_corr, int32_t* pix_to_face, void* ws, size_t ws_bytes, void* stream) {
    // every check runs before the first CUDA call
    DH_REQUIRE(bg_verts && angles_deg_host && axes_host && translations_host && R_host9 && T_host3 && target_z && corr && n_corr && ws);
    DH_REQUIRE(blur_radius >= 0.0f);
    DH_REQUIRE((reinterpret_cast<uintptr_t>(corr) & 31) == 0);      // rows are stored as one 32-byte vector
    MeshScenesPlan p;
    const int sizes = mesh_scenes_plan(n_scenes, V_bg, F_bg, V_fg, F_fg, B, scene_index, H, W, p);
    if (sizes != DH_OK) return sizes;
    DH_REQUIRE(p.F_bg <= 0 || bg_faces);
    DH_REQUIRE(p.V_fg <= 0 || (fg_verts && fg_colors));
    DH_REQUIRE(p.F_fg <= 0 || fg_faces);
    const MeshScenesLayout L = mesh_scenes_layout(n_scenes, B, p);
    if (ws_bytes < L.total) return DH_ERR_WORKSPACE;
    // the descriptor tables, uploaded as one block
    std::vector<char> tables(L.partial);
    SceneDesc* scenes_h = reinterpret_cast<SceneDesc*>(tables.data() + L.scenes);
    SceneEdit* edits_h = reinterpret_cast<SceneEdit*>(tables.data() + L.edits);
    int bg_v0 = 0, bg_f0 = 0, fg_v0 = 0, fg_f0 = 0, partial0 = 0;
    for (int s = 0; s < n_scenes; ++s) {
        SceneDesc& d = scenes_h[s];
        d.bg_v0 = bg_v0; d.V_bg = V_bg[s]; d.bg_f0 = bg_f0; d.F_bg = F_bg[s];
        d.fg_v0 = fg_v0; d.V_fg = V_fg[s]; d.fg_f0 = fg_f0; d.F_fg = F_fg[s];
        d.tp_blocks = tp_partial_blocks(V_fg[s]); d.tp_partial0 = partial0;
        d.plane = -1;
        bg_v0 += V_bg[s]; bg_f0 += F_bg[s]; fg_v0 += V_fg[s]; fg_f0 += F_fg[s]; partial0 += d.tp_blocks;
    }
    int out0 = 0, planes = 0;
    for (int b = 0; b < B; ++b) {
        SceneEdit& e = edits_h[b];
        e.scene = scene_index[b];
        e.out0 = out0;
        out0 += V_fg[e.scene];
        if (V_fg[e.scene] > 0) e.t = tp_edit(angles_deg_host[b], axes_host + 3 * b, translations_host + 3 * b);
        else e.t = TpEdit{};
        if (scenes_h[e.scene].plane < 0) {
            scenes_h[e.scene].plane = b;
            ++planes;
        }
    }
    char* w = static_cast<char*>(ws);
    const SceneDesc* scenes = reinterpret_cast<const SceneDesc*>(w + L.scenes);
    const SceneEdit* edits = reinterpret_cast<const SceneEdit*>(w + L.edits);
    double* partial = reinterpret_cast<double*>(w + L.partial);
    float* bg_ndc = reinterpret_cast<float*>(w + L.bg_ndc);
    float* fg_world = reinterpret_cast<float*>(w + L.fg_world);
    float* fg_ndc = reinterpret_cast<float*>(w + L.fg_ndc);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(w + L.keys);
    int32_t* tile_counts = reinterpret_cast<int32_t*>(w + L.tile_counts);
    const RasterCamDev cam = make_raster_cam(R_host9, T_host3, sx, sy);
    const RasterSettings st = make_raster_settings(blur_radius, cull_backfaces, perspective_correct, clip_barycentric);
    const int KS = p.KS, ntiles = p.ntiles, pair_blocks = (KS / 2 + 255) / 256;
    cudaStream_t s = as_stream(stream);
    DH_CUDA_CHECK(cudaMemcpyAsync(w, tables.data(), tables.size(), cudaMemcpyHostToDevice, s));
    // backgrounds: projected as one array, each used scene rasterised once into the plane of its first edit, copied to the others
    raster_keys_clear_kernel<<<dim3(pair_blocks, n_scenes), 256, 0, s>>>(scenes, KS, keys);
    DH_LAUNCH_CHECK();
    const int nbg = (int)p.V_bg;
    raster_project_kernel<<<(nbg + 255) / 256, 256, 0, s>>>(bg_verts, nbg, cam, bg_ndc);
    DH_LAUNCH_CHECK();
    if (p.max_F_bg > 0) {
        raster_faces_scenes_kernel<<<dim3((p.max_F_bg + 127) / 128, n_scenes), 128, 0, s>>>(bg_ndc, bg_faces, scenes, H, W, KS, st, keys);
        DH_LAUNCH_CHECK();
    }
    if (B > planes) {
        raster_keys_scenes_broadcast_kernel<<<dim3(pair_blocks, B), 256, 0, s>>>(scenes, edits, KS, keys);
        DH_LAUNCH_CHECK();
    }
    // foregrounds: every edit's transform of its scene's vertices, projected as one array, every edit's faces in one launch
    if (p.moved > 0) {
        const int rc = tp_transform_scenes(fg_verts, scenes, n_scenes, p.max_tp_blocks, edits, B, p.max_V_fg, partial, fg_world, s);
        if (rc != DH_OK) return rc;
        const int nv = (int)p.moved;
        raster_project_kernel<<<(nv + 255) / 256, 256, 0, s>>>(fg_world, nv, cam, fg_ndc);
        DH_LAUNCH_CHECK();
    }
    if (p.max_F_fg > 0) {
        raster_faces_edits_kernel<<<dim3((p.max_F_fg + 127) / 128, B), 128, 0, s>>>(fg_ndc, fg_faces, scenes, edits, H, W, KS, st, keys);
        DH_LAUNCH_CHECK();
    }
    MeshScenes m;
    m.bg_ndc = bg_ndc; m.bg_verts = bg_verts; m.bg_faces = bg_faces;
    m.fg_ndc = fg_ndc; m.fg_world = fg_world; m.fg_colors = fg_colors; m.fg_faces = fg_faces;
    m.scenes = scenes; m.edits = edits;
    const dim3 tgrid(ntiles, B);
    mesh_scenes_resolve_count_kernel<<<tgrid, kMeshTileThreads, 0, s>>>(m, keys, H, W, KS, ntiles, st, target_z, pix_to_face, tile_counts);
    DH_LAUNCH_CHECK();
    mesh_scenes_emit_kernel<<<tgrid, kMeshTileThreads, 0, s>>>(m, keys, H, W, KS, ntiles, st, tile_counts, corr, n_corr);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // namespace dh

using namespace dh;

extern "C" {

size_t dh_raster_workspace_bytes(int V, int H, int W) {
    if (V < 1 || H < 1 || W < 1) return 0;
    size_t a, b;
    return raster_layout(V, H * W, &a, &b);
}

int dh_rasterize_meshes(const float* verts, int V, const int32_t* faces, int F, int H, int W, const float* R_host9,
                        const float* T_host3, float sx, float sy, float blur_radius, int cull_backfaces, int perspective_correct,
                        int clip_barycentric, int32_t* pix_to_face, float* zbuf, float* bary, void* ws, size_t ws_bytes,
                        void* stream) {
    DH_REQUIRE(verts && faces && R_host9 && T_host3 && pix_to_face && zbuf && bary && ws);
    DH_REQUIRE(V >= 1 && F >= 0 && H >= 1 && W >= 1 && blur_radius >= 0.0f);
    size_t o_ndc, o_keys;
    if (ws_bytes < raster_layout(V, H * W, &o_ndc, &o_keys)) return DH_ERR_WORKSPACE;
    float* ndc = reinterpret_cast<float*>(static_cast<char*>(ws) + o_ndc);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(static_cast<char*>(ws) + o_keys);
    const RasterCamDev cam = make_raster_cam(R_host9, T_host3, sx, sy);
    const RasterSettings st = make_raster_settings(blur_radius, cull_backfaces, perspective_correct, clip_barycentric);
    cudaStream_t s = as_stream(stream);
    DH_CUDA_CHECK(cudaMemsetAsync(keys, 0xFF, sizeof(unsigned long long) * (size_t)H * W, s));
    raster_project_kernel<<<(V + 255) / 256, 256, 0, s>>>(verts, V, cam, ndc);
    DH_LAUNCH_CHECK();
    if (F > 0) {
        raster_faces_kernel<<<(F + 127) / 128, 128, 0, s>>>(ndc, faces, F, H, W, st, keys);
        DH_LAUNCH_CHECK();
    }
    raster_resolve_kernel<<<(H * W + 255) / 256, 256, 0, s>>>(ndc, faces, H, W, st, keys, pix_to_face, zbuf, bary);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_interpolate_face_attributes(const float* attr, int D, const int32_t* faces, const int32_t* pix_to_face, const float* bary,
                                   int H, int W, float* out, void* stream) {
    DH_REQUIRE(attr && faces && pix_to_face && bary && out && D >= 1 && H >= 1 && W >= 1);
    raster_interpolate_kernel<<<(H * W + 255) / 256, 256, 0, as_stream(stream)>>>(attr, D, faces, pix_to_face, bary, H * W, out);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

size_t dh_edit_mesh_scenes_workspace_bytes(int n_scenes, const int32_t* V_bg_host, const int32_t* F_bg_host, const int32_t* V_fg_host, const int32_t* F_fg_host,
                                           int B, const int32_t* scene_index_host, int H, int W) {
    return mesh_scenes_workspace(n_scenes, V_bg_host, F_bg_host, V_fg_host, F_fg_host, B, scene_index_host, H, W);
}

int dh_edit_mesh_scenes(int n_scenes, const float* bg_verts, const int32_t* bg_faces, const int32_t* V_bg_host, const int32_t* F_bg_host,
                        const float* fg_verts, const float* fg_colors, const int32_t* fg_faces, const int32_t* V_fg_host, const int32_t* F_fg_host,
                        int B, const int32_t* scene_index_host, const float* angles_deg_host, const float* axes_host,
                        const float* translations_host, int H, int W, const float* R_host9, const float* T_host3, float sx, float sy,
                        float blur_radius, int cull_backfaces, int perspective_correct, int clip_barycentric, float* target_z,
                        int64_t* corr, int32_t* n_corr, int32_t* pix_to_face, void* ws, size_t ws_bytes, void* stream) {
    return mesh_scenes(n_scenes, bg_verts, bg_faces, V_bg_host, F_bg_host, fg_verts, fg_colors, fg_faces, V_fg_host, F_fg_host, B, scene_index_host,
                       angles_deg_host, axes_host, translations_host, H, W, R_host9, T_host3, sx, sy, blur_radius, cull_backfaces,
                       perspective_correct, clip_barycentric, target_z, corr, n_corr, pix_to_face, ws, ws_bytes, stream);
}

size_t dh_edit_mesh_batch_workspace_bytes(int B, int V_bg, int V_fg, int H, int W) {
    if (mesh_batch_sizes(B, V_bg, 0, V_fg, 0, H, W) != DH_OK) return 0;
    return mesh_batch_layout(B, V_bg, V_fg, H, W).total;
}

int dh_edit_mesh_batch(const float* bg_verts, int V_bg, const int32_t* bg_faces, int F_bg, const float* fg_verts, const float* fg_colors,
                       int V_fg, const int32_t* fg_faces, int F_fg, int B, const float* angles_deg_host, const float* axes_host,
                       const float* translations_host, int H, int W, const float* R_host9, const float* T_host3, float sx, float sy,
                       float blur_radius, int cull_backfaces, int perspective_correct, int clip_barycentric, float* target_z,
                       int64_t* corr, int32_t* n_corr, int32_t* pix_to_face, void* ws, size_t ws_bytes, void* stream) {
    // every check runs before the first CUDA call
    DH_REQUIRE(bg_verts && angles_deg_host && axes_host && translations_host && R_host9 && T_host3 && target_z && corr && n_corr && ws);
    DH_REQUIRE(F_bg <= 0 || bg_faces);
    DH_REQUIRE(V_fg <= 0 || (fg_verts && fg_colors));
    DH_REQUIRE(F_fg <= 0 || fg_faces);
    DH_REQUIRE(blur_radius >= 0.0f);
    DH_REQUIRE((reinterpret_cast<uintptr_t>(corr) & 31) == 0);      // rows are stored as one 32-byte vector
    const int sizes = mesh_batch_sizes(B, V_bg, F_bg, V_fg, F_fg, H, W);
    if (sizes != DH_OK) return sizes;
    const MeshBatchLayout L = mesh_batch_layout(B, V_bg, V_fg, H, W);
    if (ws_bytes < L.total) return DH_ERR_WORKSPACE;
    char* w = static_cast<char*>(ws);
    double* partial = reinterpret_cast<double*>(w + L.partial);
    TpEdit* edits = reinterpret_cast<TpEdit*>(w + L.edits);
    float* bg_ndc = reinterpret_cast<float*>(w + L.bg_ndc);
    float* fg_world = reinterpret_cast<float*>(w + L.fg_world);
    float* fg_ndc = reinterpret_cast<float*>(w + L.fg_ndc);
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(w + L.keys);
    int32_t* tile_counts = reinterpret_cast<int32_t*>(w + L.tile_counts);
    const RasterCamDev cam = make_raster_cam(R_host9, T_host3, sx, sy);
    const RasterSettings st = make_raster_settings(blur_radius, cull_backfaces, perspective_correct, clip_barycentric);
    const int P = H * W, ntiles = (P + kMeshTile - 1) / kMeshTile;
    cudaStream_t s = as_stream(stream);
    std::vector<TpEdit> edits_host;
    if (V_fg > 0) {
        edits_host.resize(B);
        for (int b = 0; b < B; ++b) edits_host[b] = tp_edit(angles_deg_host[b], axes_host + 3 * b, translations_host + 3 * b);
        DH_CUDA_CHECK(cudaMemcpyAsync(edits, edits_host.data(), sizeof(TpEdit) * (size_t)B, cudaMemcpyHostToDevice, s));
    }
    // background: projected and rasterised once into edit 0's keys, then copied to the other edits
    DH_CUDA_CHECK(cudaMemsetAsync(keys, 0xFF, sizeof(unsigned long long) * (size_t)P, s));
    raster_project_kernel<<<(V_bg + 255) / 256, 256, 0, s>>>(bg_verts, V_bg, cam, bg_ndc);
    DH_LAUNCH_CHECK();
    if (F_bg > 0) {
        raster_faces_kernel<<<(F_bg + 127) / 128, 128, 0, s>>>(bg_ndc, bg_faces, F_bg, H, W, st, keys);
        DH_LAUNCH_CHECK();
    }
    if (B > 1) {
        raster_keys_broadcast_kernel<<<(P + 255) / 256, 256, 0, s>>>(keys, P, B);
        DH_LAUNCH_CHECK();
    }
    // foreground: B transforms of the same vertices, projected as one array, every edit's faces in one launch
    if (V_fg > 0) {
        const int rc = tp_transform_batch(fg_verts, V_fg, B, edits, partial, fg_world, s);
        if (rc != DH_OK) return rc;
        const int nv = B * V_fg;
        raster_project_kernel<<<(nv + 255) / 256, 256, 0, s>>>(fg_world, nv, cam, fg_ndc);
        DH_LAUNCH_CHECK();
    }
    if (F_fg > 0) {
        raster_faces_batch_kernel<<<dim3((F_fg + 127) / 128, B), 128, 0, s>>>(fg_ndc, V_fg, fg_faces, F_fg, F_bg, H, W, st, keys);
        DH_LAUNCH_CHECK();
    }
    MeshBatchScene sc;
    sc.bg_ndc = bg_ndc; sc.bg_verts = bg_verts; sc.bg_faces = bg_faces; sc.F_bg = F_bg;
    sc.fg_ndc = fg_ndc; sc.fg_world = fg_world; sc.fg_colors = fg_colors; sc.fg_faces = fg_faces; sc.V_fg = V_fg;
    const dim3 tgrid(ntiles, B);
    mesh_resolve_count_kernel<<<tgrid, kMeshTileThreads, 0, s>>>(sc, keys, H, W, ntiles, st, target_z, pix_to_face, tile_counts);
    DH_LAUNCH_CHECK();
    mesh_emit_kernel<<<tgrid, kMeshTileThreads, 0, s>>>(sc, keys, H, W, ntiles, st, tile_counts, corr, n_corr);
    DH_LAUNCH_CHECK();
    return DH_OK;
}


}  // extern "C"
