// K1: fused unproject -> rigid transform -> project (SURVEY.md 8(a) rows 2-4), plus the stand-alone
// unprojection / projection / transform_points entry points.
//
// Bit-exactness notes (SURVEY.md Appendix A): every fp32/fp64 operation below is written with the
// explicit round-to-nearest intrinsics so that nvcc can never contract a multiply-add into an FMA;
// the file is additionally compiled with -fmad=false.  The only fused operations are the two that the
// reference itself executes fused (the fp32 dot product, A.2).
#include "dh_common.cuh"

#include <math.h>
#include <string.h>

namespace dh {

thread_local int g_last_cuda_error = 0;

constexpr int kTile = 1024;          // pixels per compaction tile (small tiles: the block scans are latency bound, eight blocks per SM)
constexpr int kTileThreads = 256;    // 4 pixels per thread

struct CamDev {
    float k[9];
    float kinv[9];
    int diag;   // 1: off-diagonal entries of k and kinv are all zero (the bit-exact contract class)
};

static CamDev make_cam(const dh_camera* c) {
    CamDev d;
    memcpy(d.k, c->k, sizeof(d.k));
    memcpy(d.kinv, c->kinv, sizeof(d.kinv));
    d.diag = 1;
    for (int i = 0; i < 9; ++i)
        if (i % 4 != 0 && (c->k[i] != 0.f || c->kinv[i] != 0.f)) d.diag = 0;
    return d;
}

// depth_transform.py:634-639: p = M @ ((D * Kinv) @ [x, y, 1]^T), identity extrinsics.
__device__ __forceinline__ void unproject(const CamDev& cam, float d, float x, float y, float& X, float& Y, float& Z) {
    if (cam.diag) {
        X = -__fmul_rn(__fmul_rn(d, cam.kinv[0]), x);
        Y = -__fmul_rn(__fmul_rn(d, cam.kinv[4]), y);
        Z = __fmul_rn(__fmul_rn(d, cam.kinv[8]), 1.0f);
    } else {  // general intrinsics: left-to-right fp32 accumulation (outside the bit-exact contract)
        float r[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            float a = __fmul_rn(__fmul_rn(d, cam.kinv[3 * i + 0]), x);
            float b = __fmul_rn(__fmul_rn(d, cam.kinv[3 * i + 1]), y);
            float c = __fmul_rn(__fmul_rn(d, cam.kinv[3 * i + 2]), 1.0f);
            r[i] = __fadd_rn(__fadd_rn(a, b), c);
        }
        X = -r[0]; Y = -r[1]; Z = r[2];
    }
}

// depth_transform.py:666-687: (X,Y,Z) fp64 in pytorch3d axes -> integer pixel (u = col, v = row).
// clip to [0, size-1] first, then round half to even.  Returns false when z is NaN (never wins).
__device__ __forceinline__ bool project(const CamDev& cam, double X, double Y, double Z, int H, int W,
                                        int& u, int& v, uint64_t& key) {
    const double px = -X, py = -Y, pz = Z;
    double projx, projy, projz;
    if (cam.diag) {
        projx = __dmul_rn((double)cam.k[0], px);
        projy = __dmul_rn((double)cam.k[4], py);
        projz = __dmul_rn((double)cam.k[8], pz);
    } else {
        projx = __dadd_rn(__dadd_rn(__dmul_rn((double)cam.k[0], px), __dmul_rn((double)cam.k[1], py)), __dmul_rn((double)cam.k[2], pz));
        projy = __dadd_rn(__dadd_rn(__dmul_rn((double)cam.k[3], px), __dmul_rn((double)cam.k[4], py)), __dmul_rn((double)cam.k[5], pz));
        projz = __dadd_rn(__dadd_rn(__dmul_rn((double)cam.k[6], px), __dmul_rn((double)cam.k[7], py)), __dmul_rn((double)cam.k[8], pz));
    }
    double uu = __ddiv_rn(projx, projz);
    double vv = __ddiv_rn(projy, projz);
    const double m = (double)((H > W ? H : W) - 1);
    uu = __dmul_rn(__dadd_rn(__dmul_rn(uu, 0.5), 0.5), m);
    vv = __dmul_rn(__dadd_rn(__dmul_rn(vv, 0.5), 0.5), m);
    uu = fmin(fmax(uu, 0.0), (double)(W - 1));
    vv = fmin(fmax(vv, 0.0), (double)(H - 1));
    u = (int)rint(uu);
    v = (int)rint(vv);
    const double z = __dadd_rn(Z, 0.0);   // folds -0 into +0 (the reference compares with '<')
    key = z_to_key(z);
    return !(z != z);
}

// ------------------------------------------------------------------------------------------------
// stand-alone unprojection (depth_to_world_coords)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) unproject_kernel(const float* __restrict__ depth, int P, int W, CamDev cam,
                                                        const float* __restrict__ xs, const float* __restrict__ ys,
                                                        float* __restrict__ points) {
    const int e = blockIdx.y;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const int row = p / W, col = p - row * W;
    float X, Y, Z;
    unproject(cam, depth[(size_t)e * P + p], xs[col], ys[row], X, Y, Z);
    float* o = points + ((size_t)e * P + p) * 3;
    o[0] = X; o[1] = Y; o[2] = Z;
}

// ------------------------------------------------------------------------------------------------
// foreground compaction (raster order) + unprojection of the foreground points
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTileThreads) fg_count_kernel(const float* __restrict__ mask, int P, int ntiles,
                                                                int32_t* __restrict__ tile_counts) {
    __shared__ int warp_sums[32];
    const int e = blockIdx.y, tile = blockIdx.x;
    const int p0 = tile * kTile + threadIdx.x * 4;
    const float* m = mask + (size_t)e * P;
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (p0 + i < P && m[p0 + i] != 0.0f) ++c;
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if (lane_id() == 0) warp_sums[warp_id()] = c;
    __syncthreads();
    if (warp_id() == 0) {
        int s = lane_id() < (int)(blockDim.x >> 5) ? warp_sums[lane_id()] : 0;
        s = __reduce_add_sync(0xFFFFFFFFu, s);
        if (lane_id() == 0) tile_counts[e * ntiles + tile] = s;
    }
}

// `points` != nullptr: the foreground points are taken from an (P,3) fp32 array instead of being unprojected
// from `depth` (transform_point_cloud entry point).
__global__ void __launch_bounds__(kTileThreads) fg_compact_kernel(
    const float* __restrict__ depth, const float* __restrict__ mask, int P, int W, int ntiles, CamDev cam,
    const float* __restrict__ xs, const float* __restrict__ ys, const int32_t* __restrict__ tile_counts,
    int32_t* __restrict__ fg_index, float* __restrict__ fgX, float* __restrict__ fgY, float* __restrict__ fgZ,
    int32_t* __restrict__ n_fg, const float* __restrict__ points) {
    __shared__ int scan_smem[33];
    __shared__ int base_smem;
    const int e = blockIdx.y, tile = blockIdx.x;
    // base = number of foreground pixels in the preceding tiles of this edit
    int part = 0;
    for (int t = threadIdx.x; t < tile; t += blockDim.x) part += tile_counts[e * ntiles + t];
    int tot;
    block_exclusive_scan(part, scan_smem, tot);
    if (threadIdx.x == 0) base_smem = tot;
    __syncthreads();
    const int base = base_smem;

    const int p0 = tile * kTile + threadIdx.x * 4;
    const float* m = mask + (size_t)e * P;
    bool f[4];
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        f[i] = (p0 + i < P) && (m[p0 + i] != 0.0f);
        c += f[i];
    }
    int total;
    int pos = base + block_exclusive_scan(c, scan_smem, total);
    const size_t eo = (size_t)e * P;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!f[i]) continue;
        const int p = p0 + i;
        const int row = p / W, col = p - row * W;
        float X, Y, Z;
        if (points) {
            X = points[3 * (eo + p)]; Y = points[3 * (eo + p) + 1]; Z = points[3 * (eo + p) + 2];
        } else {
            unproject(cam, depth[eo + p], xs[col], ys[row], X, Y, Z);
        }
        fg_index[eo + pos] = p;
        fgX[eo + pos] = X; fgY[eo + pos] = Y; fgZ[eo + pos] = Z;
        ++pos;
    }
    if (tile == ntiles - 1 && threadIdx.x == 0) n_fg[e] = base + total;
}

// Sequential fp32 sum in raster order, one warp per component (np.mean(points[mask], axis=0) adds row
// by row, depth_transform.py:509).  All 32 lanes carry the same running sum.  The addends are staged in
// shared memory 512 at a time with asynchronous copies (a ring of tiles per warp) and read back with 128-bit
// broadcast loads into a REGISTER double buffer of 32 values: while the dependent FADD chain (4 cycles per
// element) works through one group, the loads of the next group are already in flight.
__global__ void __launch_bounds__(96) fg_centroid_kernel(const float* __restrict__ fgX, const float* __restrict__ fgY,
                                                         const float* __restrict__ fgZ, const int32_t* __restrict__ n_fg,
                                                         int P, float* __restrict__ centroid) {
    constexpr int kTileF = 512, kBuf = 4, kGroup = 8;            // floats per tile, ring depth, float4 per register group
    __shared__ __align__(16) float ring[3][kBuf][kTileF];
    const int e = blockIdx.x, comp = warp_id(), lane = lane_id();
    const float* a = (comp == 0 ? fgX : comp == 1 ? fgY : fgZ) + (size_t)e * P;   // 256-byte aligned (workspace layout)
    const int n = n_fg[e];
    const unsigned full = 0xFFFFFFFFu;
    float s = 0.0f;
    const int n_tiles = (reinterpret_cast<uintptr_t>(a) & 15) == 0 ? n / kTileF : 0;
    auto issue = [&](int t) {
        if (t < n_tiles) {
            const float* src = a + (size_t)t * kTileF + lane * 4;
            float* dst = &ring[comp][t % kBuf][lane * 4];
#pragma unroll
            for (int q = 0; q < kTileF / 128; ++q)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst + 128 * q)),
                             "l"(src + 128 * q) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");       // (empty groups keep the wait count uniform)
    };
#pragma unroll
    for (int t = 0; t < kBuf - 1; ++t) issue(t);
    for (int t = 0; t < n_tiles; ++t) {
        issue(t + kBuf - 1);                                        // refills the slot consumed in iteration t - 1
        asm volatile("cp.async.wait_group %0;" ::"n"(kBuf - 1) : "memory");
        __syncwarp();
        const float4* tile = reinterpret_cast<const float4*>(ring[comp][t % kBuf]);
        float4 cur[kGroup], nxt[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) cur[j] = tile[j];          // same address in every lane: broadcast
#pragma unroll
        for (int g = 0; g < kTileF / 4 / kGroup; ++g) {
            if (g + 1 < kTileF / 4 / kGroup) {
#pragma unroll
                for (int j = 0; j < kGroup; ++j) nxt[j] = tile[(g + 1) * kGroup + j];
            }
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                s = __fadd_rn(s, cur[j].x);
                s = __fadd_rn(s, cur[j].y);
                s = __fadd_rn(s, cur[j].z);
                s = __fadd_rn(s, cur[j].w);
            }
#pragma unroll
            for (int j = 0; j < kGroup; ++j) cur[j] = nxt[j];
        }
        __syncwarp();                                               // every lane is done with the slot before it is refilled
    }
    for (int base = n_tiles * kTileF; base < n; base += 32) {
        const float v = base + lane < n ? a[base + lane] : 0.0f;
        const int cnt = min(32, n - base);
        for (int j = 0; j < cnt; ++j) s = __fadd_rn(s, __shfl_sync(full, v, j));
    }
    if (lane == 0) centroid[e * 3 + comp] = __fdiv_rn(s, (float)n);
}

constexpr int kSeqTileF = 512, kSeqBuf = 4;                      // floats per tile, ring depth
using SeqRing = float[3][kSeqBuf][kSeqTileF];

// The FADD chain of fg_centroid_kernel as a function of its own (fg_centroid_kernel keeps its inline copy, and with it its exact
// instruction schedule): the sequential fp32 sum of a[0..n) by warp `comp`, staged in ring[comp], every lane holding the sum.
__device__ __forceinline__ float seq_sum_warp(const float* __restrict__ a, int n, int comp, int lane, SeqRing& ring) {
    constexpr int kTileF = kSeqTileF, kBuf = kSeqBuf, kGroup = 8;   // float4 per register group
    const unsigned full = 0xFFFFFFFFu;
    float s = 0.0f;
    const int n_tiles = (reinterpret_cast<uintptr_t>(a) & 15) == 0 ? n / kTileF : 0;
    auto issue = [&](int t) {
        if (t < n_tiles) {
            const float* src = a + (size_t)t * kTileF + lane * 4;
            float* dst = &ring[comp][t % kBuf][lane * 4];
#pragma unroll
            for (int q = 0; q < kTileF / 128; ++q)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst + 128 * q)),
                             "l"(src + 128 * q) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");       // (empty groups keep the wait count uniform)
    };
#pragma unroll
    for (int t = 0; t < kBuf - 1; ++t) issue(t);
    for (int t = 0; t < n_tiles; ++t) {
        issue(t + kBuf - 1);                                        // refills the slot consumed in iteration t - 1
        asm volatile("cp.async.wait_group %0;" ::"n"(kBuf - 1) : "memory");
        __syncwarp();
        const float4* tile = reinterpret_cast<const float4*>(ring[comp][t % kBuf]);
        float4 cur[kGroup], nxt[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) cur[j] = tile[j];          // same address in every lane: broadcast
#pragma unroll
        for (int g = 0; g < kTileF / 4 / kGroup; ++g) {
            if (g + 1 < kTileF / 4 / kGroup) {
#pragma unroll
                for (int j = 0; j < kGroup; ++j) nxt[j] = tile[(g + 1) * kGroup + j];
            }
#pragma unroll
            for (int j = 0; j < kGroup; ++j) {
                s = __fadd_rn(s, cur[j].x);
                s = __fadd_rn(s, cur[j].y);
                s = __fadd_rn(s, cur[j].z);
                s = __fadd_rn(s, cur[j].w);
            }
#pragma unroll
            for (int j = 0; j < kGroup; ++j) cur[j] = nxt[j];
        }
        __syncwarp();                                               // every lane is done with the slot before it is refilled
    }
    for (int base = n_tiles * kTileF; base < n; base += 32) {
        const float v = base + lane < n ? a[base + lane] : 0.0f;
        const int cnt = min(32, n - base);
        for (int j = 0; j < cnt; ++j) s = __fadd_rn(s, __shfl_sync(full, v, j));
    }
    return s;
}

// depth_transform.py:512-531 for one point: Rodrigues about the centroid + translation, fp32 -> fp64 in the
// reference's operation order (SURVEY.md A.2).
__device__ __forceinline__ void rigid_point(float px, float py, float pz, float cx, float cy, float cz, const dh_rigid& rg,
                                            double& X, double& Y, double& Z) {
    const float qx = __fsub_rn(px, cx), qy = __fsub_rn(py, cy), qz = __fsub_rn(pz, cz);
    const float ax = rg.axis[0], ay = rg.axis[1], az = rg.axis[2];
    const float crx = __fsub_rn(__fmul_rn(ay, qz), __fmul_rn(az, qy));
    const float cry = __fsub_rn(__fmul_rn(az, qx), __fmul_rn(ax, qz));
    const float crz = __fsub_rn(__fmul_rn(ax, qy), __fmul_rn(ay, qx));
    float d = __fmul_rn(qy, ay);
    d = __fmaf_rn(qx, ax, d);
    d = __fmaf_rn(qz, az, d);
    const float t3x = __fmul_rn(ax, d), t3y = __fmul_rn(ay, d), t3z = __fmul_rn(az, d);
    const double c = rg.cos_t, s = rg.sin_t, omc = __dsub_rn(1.0, c);
    X = __dadd_rn(__dadd_rn(__dmul_rn((double)qx, c), __dmul_rn((double)crx, s)), __dmul_rn((double)t3x, omc));
    Y = __dadd_rn(__dadd_rn(__dmul_rn((double)qy, c), __dmul_rn((double)cry, s)), __dmul_rn((double)t3y, omc));
    Z = __dadd_rn(__dadd_rn(__dmul_rn((double)qz, c), __dmul_rn((double)crz, s)), __dmul_rn((double)t3z, omc));
    X = __dadd_rn(__dadd_rn(X, (double)cx), rg.t[0]);
    Y = __dadd_rn(__dadd_rn(Y, (double)cy), rg.t[1]);
    Z = __dadd_rn(__dadd_rn(Z, (double)cz), rg.t[2]);
}

__global__ void __launch_bounds__(256) rigid_all_kernel(const float* __restrict__ points, int N, const dh_rigid* __restrict__ rigid,
                                                        const float* __restrict__ centroid, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double X, Y, Z;
    rigid_point(points[3 * (size_t)i], points[3 * (size_t)i + 1], points[3 * (size_t)i + 2], centroid[0], centroid[1], centroid[2],
                rigid[0], X, Y, Z);
    out[3 * (size_t)i] = X; out[3 * (size_t)i + 1] = Y; out[3 * (size_t)i + 2] = Z;
}

// ------------------------------------------------------------------------------------------------
// The edit fast path: K1 + K2 of a batch of edits in seven launches, no memsets, built on one fact:
//
//   a background point keeps its pixel.  With the library's pinhole camera (diagonal K, principal point 0, square image)
//   the point unprojected from pixel (r, c) projects back to (u, v) = (c, r) exactly: the fp32 roundings of the
//   unprojection and the fp32 K^-1 move u by less than (S / 2) * 3e-7 pixels (SURVEY.md A.1 / A.4), far from a rounding
//   boundary of rint().  So the z-buffer can be INITIALISED with the keys of the background depths (plain coalesced stores
//   instead of a memset plus 2^18 64-bit atomics per edit), the fp64 transform / projection with its two IEEE divisions runs
//   for the n_fg foreground points only, and a background pixel resolves itself: it wins iff its own key is still in the
//   z-buffer (its index is the lowest of all points that can reach the pixel, so it also wins exact z ties).
//
// Background depths outside the "nice" class - zero, infinite, subnormal or absurdly large magnitudes, or any depth when the
// camera / image is not of the class above - are not trusted: those pixels are appended to a per-edit list of ODD points that
// travel through the generic path together with the foreground points (index < P, so they keep their rank in ties).  NaN
// depths never reach the z-buffer at all (depth_transform.py:697-712: a NaN never satisfies '<').  Results are bit-identical
// in every case to dh_splat_zbuffer + dh_splat_resolve over the generic pixel / key of every point (the debug outputs below
// record them for the background points too).
// ------------------------------------------------------------------------------------------------
struct EditWs {
    int32_t* tile_counts;
    dh_rigid* rigid;
    float *fgX, *fgY, *fgZ;
    int32_t* odd_list;      // [B][P] pixels whose background point takes the generic path
    int32_t* odd_count;     // [B]
    uint32_t* minmax_keys;  // [B][4] order-preserving keys: min / -max of the non-negative depths, min / -max of the negative ones
};

__device__ __forceinline__ bool nice_depth(float d) {
    const float a = fabsf(d);
    return a >= 1e-30f && a <= 1e30f;         // (false for NaN)
}

__device__ __forceinline__ uint64_t bg_key(float d) { return z_to_key(__dadd_rn((double)d, 0.0)); }     // Z = d (k[8] = 1), -0 folded

// A: foreground counts per tile (for the compaction) + z-buffer initialised with the background keys, 4 pixels per thread.
__global__ void __launch_bounds__(kTileThreads) edit_prepare_kernel(
    const float* __restrict__ mask, const float* __restrict__ bg_depth, int P, int W, int H, int ntiles, int cam_nice, CamDev cam,
    const float* __restrict__ xs, const float* __restrict__ ys,
    int32_t* __restrict__ tile_counts, uint64_t* __restrict__ zbuf, EditWs ws,
    int32_t* __restrict__ dbg_pix, uint64_t* __restrict__ dbg_zkey, double* __restrict__ dbg_points) {
    __shared__ int warp_sums[32];
    const int e = blockIdx.y, tile = blockIdx.x;
    const int p0 = tile * kTile + threadIdx.x * 4;
    const size_t eo = (size_t)e * P;
    if (tile == 0 && threadIdx.x < 4) ws.minmax_keys[e * 4 + threadIdx.x] = 0xFFFFFFFFu;      // (all four are kept as minima)
    float m4[4] = {0.f, 0.f, 0.f, 0.f}, d4[4] = {0.f, 0.f, 0.f, 0.f};
    const bool vec = p0 + 3 < P && ((eo + p0) & 3) == 0;
    if (vec) {
        const float4 mv = __ldg(reinterpret_cast<const float4*>(mask + eo + p0));
        const float4 dv = __ldg(reinterpret_cast<const float4*>(bg_depth + eo + p0));
        m4[0] = mv.x; m4[1] = mv.y; m4[2] = mv.z; m4[3] = mv.w;
        d4[0] = dv.x; d4[1] = dv.y; d4[2] = dv.z; d4[3] = dv.w;
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (p0 + i < P) { m4[i] = mask[eo + p0 + i]; d4[i] = bg_depth[eo + p0 + i]; }
    }
    int c = 0;
    uint64_t k4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        k4[i] = kEmptyZ;
        if (p0 + i >= P) continue;
        c += m4[i] != 0.0f;
        const float d = d4[i];
        if (cam_nice && nice_depth(d)) {
            k4[i] = bg_key(d);
        } else if (d == d) {                       // odd point: generic path (kernels D, F, G); NaN: no candidate at all
            ws.odd_list[eo + atomicAdd(ws.odd_count + e, 1)] = p0 + i;
        }
        if (dbg_pix) {                             // debug outputs: the generic projection of EVERY background point
            const int p = p0 + i, row = p / W, col = p - row * W;
            float x, y, z;
            unproject(cam, d, xs[col], ys[row], x, y, z);
            int u, v;
            uint64_t key;
            const bool ok = project(cam, (double)x, (double)y, (double)z, H, W, u, v, key);
            dbg_pix[(size_t)e * 2 * P + p] = ok ? v * W + u : -1;
            dbg_zkey[(size_t)e * 2 * P + p] = key;
            if (dbg_points) {
                double* o = dbg_points + ((size_t)e * 2 * P + p) * 3;
                o[0] = (double)x; o[1] = (double)y; o[2] = (double)z;
            }
        }
    }
    if (vec) {
        ulonglong2* zb = reinterpret_cast<ulonglong2*>(zbuf + eo + p0);
        zb[0] = make_ulonglong2(k4[0], k4[1]);
        zb[1] = make_ulonglong2(k4[2], k4[3]);
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (p0 + i < P) zbuf[eo + p0 + i] = k4[i];
    }
    c = __reduce_add_sync(0xFFFFFFFFu, c);
    if (lane_id() == 0) warp_sums[warp_id()] = c;
    __syncthreads();
    if (warp_id() == 0) {
        int s = lane_id() < (int)(blockDim.x >> 5) ? warp_sums[lane_id()] : 0;
        s = __reduce_add_sync(0xFFFFFFFFu, s);
        if (lane_id() == 0) tile_counts[e * ntiles + tile] = s;
    }
}

// generic point of the edit: slot < n_fg -> foreground point `slot` (index P + slot); then the odd background points
struct EditPoint {
    bool live;
    int index;       // point index in the reference's order (background p, foreground P + j)
    double X, Y, Z;
};

__device__ __forceinline__ EditPoint edit_point(int e, int slot, int P, int W, const CamDev& cam, const dh_rigid* __restrict__ rigid,
                                                const float* __restrict__ xs, const float* __restrict__ ys,
                                                const float* __restrict__ bg_depth, const int32_t* __restrict__ n_fg,
                                                const float* __restrict__ centroid, const EditWs& ws) {
    EditPoint pt;
    pt.live = false; pt.index = -1; pt.X = pt.Y = pt.Z = 0.0;
    const int nf = n_fg[e];
    if (slot < nf) {
        const size_t eo = (size_t)e * P + slot;
        rigid_point(ws.fgX[eo], ws.fgY[eo], ws.fgZ[eo], centroid[e * 3 + 0], centroid[e * 3 + 1], centroid[e * 3 + 2], rigid[e], pt.X, pt.Y, pt.Z);
        pt.live = true; pt.index = P + slot;
    } else if (slot - nf < ws.odd_count[e]) {
        const int p = ws.odd_list[(size_t)e * P + (slot - nf)];
        const int row = p / W, col = p - row * W;
        float x, y, z;
        unproject(cam, bg_depth[(size_t)e * P + p], xs[col], ys[row], x, y, z);
        pt.X = (double)x; pt.Y = (double)y; pt.Z = (double)z;
        pt.live = true; pt.index = p;
    }
    return pt;
}

__device__ __forceinline__ int generic_index(int e, int slot, int P, const int32_t* __restrict__ n_fg, const EditWs& ws) {
    const int nf = n_fg[e];
    if (slot < nf) return P + slot;
    return slot - nf < ws.odd_count[e] ? ws.odd_list[(size_t)e * P + (slot - nf)] : -1;
}

// D: generic points: transform / project, record pixel and key, pass 1 of the splat (64-bit atomicMin on the z key)
__global__ void __launch_bounds__(256) edit_points_splat_kernel(
    const float* __restrict__ bg_depth, int P, int H, int W, CamDev cam, const dh_rigid* __restrict__ rigid,
    const float* __restrict__ xs, const float* __restrict__ ys, const int32_t* __restrict__ n_fg, const float* __restrict__ centroid,
    EditWs ws, int32_t* __restrict__ pix, uint64_t* __restrict__ zkey, double* __restrict__ dbg_points, uint64_t* zbuf) {
    const int e = blockIdx.y;
    const int n = n_fg[e] + ws.odd_count[e];
    uint64_t* zb = zbuf + (size_t)e * P;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {      // (block-stride: n is only known here)
        const int slot = base + threadIdx.x;
        const EditPoint pt = edit_point(e, slot, P, W, cam, rigid, xs, ys, bg_depth, n_fg, centroid, ws);
        int q = -1;
        uint64_t key = kEmptyZ;
        if (pt.live) {
            int u, v;
            const bool ok = project(cam, pt.X, pt.Y, pt.Z, H, W, u, v, key);
            q = ok ? v * W + u : -1;
            // pixel and key are kept at the point's own index (background p, foreground P + j): passes F and G and the
            // correspondences read them back from there
            const size_t po = (size_t)e * 2 * P + pt.index;
            pix[po] = q; zkey[po] = key;
            if (dbg_points) {
                double* o = dbg_points + po * 3;
                o[0] = pt.X; o[1] = pt.Y; o[2] = pt.Z;
            }
        }
        zbuf_atomic_min_warp(zb, q, key);
    }
}

// E: every pixel resolves what it can: depth map, target mask, and - when its own (nice) background point holds the z-buffer
// entry - the winner.  One warp per 32-pixel word of a row (the ballot packs the mask), block-stride over the words of an edit.
__global__ void __launch_bounds__(256) edit_resolve_kernel(
    const uint64_t* __restrict__ zbuf, const float* __restrict__ bg_depth, int H, int W, int wpr, int cam_nice,
    uint32_t* __restrict__ winner, float* __restrict__ depth_map, uint8_t* __restrict__ target_mask, uint32_t* __restrict__ target_bits,
    int32_t* __restrict__ winner_src, EditWs ws) {
    __shared__ float red[4][8];
    const int e = blockIdx.y;
    const int P = H * W, words = H * wpr;
    const float inf = __int_as_float(0x7F800000);
    float r[4] = {inf, inf, inf, inf};      // min(d >= 0), -max(d >= 0), min(d < 0), -max(d < 0): all kept as minima
    for (int word = blockIdx.x * (blockDim.x >> 5) + warp_id(); word < words; word += gridDim.x * (blockDim.x >> 5)) {
        const int row = word / wpr, col = (word - row * wpr) * 32 + lane_id();
        bool fg = false;
        if (col < W) {
            const int p = row * W + col;
            const size_t q = (size_t)e * P + p;
            const uint64_t z = zbuf[q];
            const float bd = bg_depth[q];
            float d = inf;                                        // +inf: empty pixel (depth_transform.py:689)
            uint32_t w = kNoWinner;
            if (z != kEmptyZ) {
                d = __double2float_rn(key_to_z(z));
                if (cam_nice && nice_depth(bd) && bg_key(bd) == z) w = (uint32_t)p;   // own background point: lowest index, wins ties
                else fg = true;      // provisional: a generic point holds the entry (foreground unless an odd background point wins)
            }
            winner[q] = w;
            depth_map[q] = d;
            if (winner_src) winner_src[q] = w == kNoWinner ? -1 : (int32_t)p;
            if (target_mask) target_mask[q] = fg ? 1 : 0;
            if (d == d) {
                if (__float_as_uint(d) & 0x80000000u) { r[2] = fminf(r[2], d); r[3] = fminf(r[3], -d); }
                else { r[0] = fminf(r[0], d); r[1] = fminf(r[1], -d); }
            }
        }
        const uint32_t bits = __ballot_sync(0xFFFFFFFFu, fg);
        if (lane_id() == 0) target_bits[(size_t)e * words + word] = bits;
    }
    // min / max of the depth map for normalize_depth(1 / depth): block reduction, then one atomic per block and extremum on
    // order-preserving keys (min / max do not depend on the order: deterministic)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r[k] = fminf(r[k], __shfl_xor_sync(0xFFFFFFFFu, r[k], o));
        if (lane_id() == 0) red[k][warp_id()] = r[k];
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        float v = inf;
        for (int w8 = 0; w8 < (int)(blockDim.x >> 5); ++w8) v = fminf(v, red[threadIdx.x][w8]);
        red[threadIdx.x][0] = v;
    }
    __syncthreads();
    // (a group is present iff its "-max" / "min" slot left +inf: -d <= 0 for d >= 0, d < 0 otherwise; +inf depths of empty pixels count)
    if (threadIdx.x == 0) {
        if (red[1][0] != inf) { atomicMin(ws.minmax_keys + e * 4 + 0, f_to_key(red[0][0])); atomicMin(ws.minmax_keys + e * 4 + 1, f_to_key(red[1][0])); }
        if (red[2][0] != inf) { atomicMin(ws.minmax_keys + e * 4 + 2, f_to_key(red[2][0])); atomicMin(ws.minmax_keys + e * 4 + 3, f_to_key(red[3][0])); }
    }
}

// F: pass 2 of the splat for the generic points: among the points whose key equals the z-buffer entry the lowest index wins
__global__ void __launch_bounds__(256) edit_points_winner_kernel(
    const int32_t* __restrict__ pix, const uint64_t* __restrict__ zkey,
    const int32_t* __restrict__ n_fg, int P, const uint64_t* __restrict__ zbuf, uint32_t* winner, EditWs ws) {
    const int e = blockIdx.y;
    const int n = n_fg[e] + ws.odd_count[e];
    uint32_t* wb = winner + (size_t)e * P;
    const unsigned full = 0xFFFFFFFFu;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int slot = base + threadIdx.x;
        int q = -1;
        bool tie = false;
        uint32_t idx = kNoWinner;
        if (slot < n) {
            const int index = generic_index(e, slot, P, n_fg, ws);
            const size_t go = (size_t)e * 2 * P + index;
            q = pix[go];
            if (q >= 0) tie = zkey[go] == zbuf[(size_t)e * P + q];
            idx = (uint32_t)index;
        }
        const int q0 = __shfl_sync(full, q, 0);
        if (__all_sync(full, q == q0)) {
            if (q0 >= 0) {
                const uint32_t m = __reduce_min_sync(full, tie ? idx : kNoWinner);
                if (lane_id() == 0 && m != kNoWinner && m < *(volatile uint32_t*)(wb + q0)) atomicMin(wb + q0, m);
            }
        } else if (tie && idx < *(volatile uint32_t*)(wb + q)) {
            atomicMin(wb + q, idx);
        }
    }
}

// G: the generic points that won their pixel publish themselves (source pixel of the winner; an odd BACKGROUND winner also
// clears the provisional foreground bit), and the first thread of every edit finishes the min / max of 1 / depth.
__global__ void __launch_bounds__(256) edit_points_publish_kernel(
    const int32_t* __restrict__ pix, const int32_t* __restrict__ n_fg,
    const int32_t* __restrict__ fg_index, int P, int W, int wpr, const uint32_t* __restrict__ winner, int32_t* __restrict__ winner_src,
    uint8_t* __restrict__ target_mask, uint32_t* __restrict__ target_bits, EditWs ws, float* __restrict__ inv_minmax) {
    const int e = blockIdx.y;
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot == 0 && inv_minmax) {
        // IEEE division is monotone: min / max of fl(1/d) from the four extrema of d (bit-identical to reducing fl(1/d))
        const float inf = __int_as_float(0x7F800000);
        const uint32_t* k = ws.minmax_keys + e * 4;
        float mn = inf, mx = -inf;
        if (k[1] != 0xFFFFFFFFu) {          // some non-negative depth: reciprocals in [1/pmax, 1/pmin]
            mn = fminf(mn, __fdiv_rn(1.0f, -key_to_f(k[1])));
            mx = fmaxf(mx, __fdiv_rn(1.0f, key_to_f(k[0])));
        }
        if (k[2] != 0xFFFFFFFFu) {          // some negative depth: reciprocals in [1/nmax, 1/nmin]
            mn = fminf(mn, __fdiv_rn(1.0f, -key_to_f(k[3])));
            mx = fmaxf(mx, __fdiv_rn(1.0f, key_to_f(k[2])));
        }
        inv_minmax[e * 2] = mn;
        inv_minmax[e * 2 + 1] = mx;
    }
    const int n = n_fg[e] + ws.odd_count[e];
    for (int sl = slot; sl < n; sl += gridDim.x * blockDim.x) {
        const int index = generic_index(e, sl, P, n_fg, ws);
        const int q = pix[(size_t)e * 2 * P + index];
        if (q < 0) continue;
        const uint32_t idx = (uint32_t)index;
        if (winner[(size_t)e * P + q] != idx) continue;
        if ((int)idx >= P) {
            if (winner_src) winner_src[(size_t)e * P + q] = fg_index[(size_t)e * P + (idx - P)];
        } else {                                // an odd background point won: not foreground after all
            if (winner_src) winner_src[(size_t)e * P + q] = (int32_t)idx;
            if (target_mask) target_mask[(size_t)e * P + q] = 0;
            const int row = q / W, col = q - row * W;
            atomicAnd(target_bits + (size_t)e * (P / W) * wpr + row * wpr + (col >> 5), ~(1u << (col & 31)));
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Multi-object edits (dh_edit_splat_objects): the foreground is the union of K <= 16 disjoint objects, labels[p] = k + 1 for
// a pixel of object k.  The compaction of the union also records each foreground point's object; every point then moves about
// the sequential centroid of its own object with its object's rigid transform.  The z-buffer, masks and winners do not depend on
// which object a point came from: kernels A, E, F and G run unchanged.
// ------------------------------------------------------------------------------------------------
constexpr int kMaxObjects = 16;

struct ObjWs {
    int32_t* tile_hist;         // [B][ntiles][16]: foreground pixels of each object in each compaction tile
    float *objX, *objY, *objZ;  // [B][stride]: the points of each object compacted, object k from a 16-byte aligned offset
    size_t stride;
};

// B: the union compaction of fg_compact_kernel, plus the object of every foreground point and per-tile object counts.
__global__ void __launch_bounds__(kTileThreads) fg_compact_objects_kernel(
    const float* __restrict__ depth, const float* __restrict__ mask, const uint8_t* __restrict__ labels, int P, int W, int ntiles,
    int K, CamDev cam, const float* __restrict__ xs, const float* __restrict__ ys, const int32_t* __restrict__ tile_counts,
    int32_t* __restrict__ fg_index, uint8_t* __restrict__ fg_object, float* __restrict__ fgX, float* __restrict__ fgY,
    float* __restrict__ fgZ, int32_t* __restrict__ n_fg, int32_t* __restrict__ tile_hist) {
    __shared__ int scan_smem[33];
    __shared__ int base_smem;
    __shared__ int hist[kMaxObjects];
    const int e = blockIdx.y, tile = blockIdx.x;
    if (threadIdx.x < kMaxObjects) hist[threadIdx.x] = 0;
    int part = 0;
    for (int t = threadIdx.x; t < tile; t += blockDim.x) part += tile_counts[e * ntiles + t];
    int tot;
    block_exclusive_scan(part, scan_smem, tot);
    if (threadIdx.x == 0) base_smem = tot;
    __syncthreads();
    const int base = base_smem;

    const int p0 = tile * kTile + threadIdx.x * 4;
    const float* m = mask + (size_t)e * P;
    bool f[4];
    int c = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        f[i] = (p0 + i < P) && (m[p0 + i] != 0.0f);
        c += f[i];
    }
    int total;
    int pos = base + block_exclusive_scan(c, scan_smem, total);
    const size_t eo = (size_t)e * P;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if (!f[i]) continue;
        const int p = p0 + i;
        const int row = p / W, col = p - row * W;
        float X, Y, Z;
        unproject(cam, depth[eo + p], xs[col], ys[row], X, Y, Z);
        // (a foreground pixel whose label is 0 or above K - the caller broke the contract - is taken as object K - 1)
        const int k = min((int)(uint8_t)(labels[eo + p] - 1u), K - 1);
        fg_index[eo + pos] = p;
        fg_object[eo + pos] = (uint8_t)k;
        fgX[eo + pos] = X; fgY[eo + pos] = Y; fgZ[eo + pos] = Z;
        atomicAdd(&hist[k], 1);
        ++pos;
    }
    __syncthreads();
    if (threadIdx.x < kMaxObjects) tile_hist[((size_t)e * ntiles + tile) * kMaxObjects + threadIdx.x] = hist[threadIdx.x];
    if (tile == ntiles - 1 && threadIdx.x == 0) n_fg[e] = base + total;
}

// C: the sequential centroid of object k = blockIdx.x of edit e = blockIdx.y.  The block first copies the object's points out
// of the compacted union (a raster-ordered subsequence, found by a block scan over the object ids), then three warps run the
// FADD chain of fg_centroid_kernel over that object alone: the chain is as long as the object, not the union.
__global__ void __launch_bounds__(256) fg_centroid_objects_kernel(const float* __restrict__ fgX, const float* __restrict__ fgY,
                                                                  const float* __restrict__ fgZ, const uint8_t* __restrict__ fg_object,
                                                                  const int32_t* __restrict__ n_fg, int P, int ntiles, int K, ObjWs ow,
                                                                  float* __restrict__ centroid) {
    __shared__ __align__(16) float ring[3][kSeqBuf][kSeqTileF];
    __shared__ int counts[8][kMaxObjects];
    __shared__ int scan_smem[33];
    const int k = blockIdx.x, e = blockIdx.y;
    // points per object of this edit: the sums of the tile histograms (64-byte rows)
    int c[kMaxObjects];
#pragma unroll
    for (int j = 0; j < kMaxObjects; ++j) c[j] = 0;
    for (int t = threadIdx.x; t < ntiles; t += blockDim.x) {
        const int4* h = reinterpret_cast<const int4*>(ow.tile_hist + ((size_t)e * ntiles + t) * kMaxObjects);
#pragma unroll
        for (int q = 0; q < kMaxObjects / 4; ++q) {
            const int4 v = h[q];
            c[4 * q] += v.x; c[4 * q + 1] += v.y; c[4 * q + 2] += v.z; c[4 * q + 3] += v.w;
        }
    }
#pragma unroll
    for (int j = 0; j < kMaxObjects; ++j) {
        const int s = __reduce_add_sync(0xFFFFFFFFu, c[j]);
        if (lane_id() == 0) counts[warp_id()][j] = s;
    }
    __syncthreads();
    int n_k = 0, off = 0;                       // object k's count and its 16-byte aligned offset in the object arrays
    for (int j = 0; j <= k; ++j) {
        int nj = 0;
        for (int w = 0; w < 8; ++w) nj += counts[w][j];
        if (j < k) off += (nj + 3) & ~3;
        else n_k = nj;
    }
    const size_t eo = (size_t)e * P;
    float* dx = ow.objX + e * ow.stride + off;
    float* dy = ow.objY + e * ow.stride + off;
    float* dz = ow.objZ + e * ow.stride + off;
    const int n = n_fg[e];
    // stable compaction of the object's points, 4096 union points per step (16 id loads in flight per thread), until all n_k are found
    constexpr int kPer = 16;
    for (int base = 0, found = 0; found < n_k && base < n; base += kPer * 256) {
        const int j0 = base + threadIdx.x * kPer;
        uint32_t f = 0;
#pragma unroll
        for (int i = 0; i < kPer; ++i)
            if (j0 + i < n && fg_object[eo + j0 + i] == k) f |= 1u << i;
        int total;
        int q = found + block_exclusive_scan(__popc(f), scan_smem, total);
        for (; f; f &= f - 1) {
            const size_t j = eo + j0 + __ffs(f) - 1;
            dx[q] = fgX[j]; dy[q] = fgY[j]; dz[q] = fgZ[j];
            ++q;
        }
        found += total;
    }
    __syncthreads();                            // the block's global writes are visible to its own warps
    const int comp = warp_id();
    if (comp < 3) {
        const float s = seq_sum_warp(comp == 0 ? dx : comp == 1 ? dy : dz, n_k, comp, lane_id(), ring);
        if (lane_id() == 0) centroid[((size_t)e * K + k) * 3 + comp] = __fdiv_rn(s, (float)n_k);
    }
}

// a generic point of a multi-object edit: a foreground point moves with its own object's centroid and transform
__device__ __forceinline__ EditPoint edit_point_objects(int e, int slot, int P, int W, int K, const CamDev& cam,
                                                        const dh_rigid* __restrict__ rigid, const float* __restrict__ xs,
                                                        const float* __restrict__ ys, const float* __restrict__ bg_depth,
                                                        const int32_t* __restrict__ n_fg, const uint8_t* __restrict__ fg_object,
                                                        const float* __restrict__ centroid, const EditWs& ws) {
    if (slot < n_fg[e]) {
        EditPoint pt;
        const size_t eo = (size_t)e * P + slot;
        const int ek = e * K + fg_object[eo];
        rigid_point(ws.fgX[eo], ws.fgY[eo], ws.fgZ[eo], centroid[ek * 3 + 0], centroid[ek * 3 + 1], centroid[ek * 3 + 2], rigid[ek],
                    pt.X, pt.Y, pt.Z);
        pt.live = true; pt.index = P + slot;
        return pt;
    }
    return edit_point(e, slot, P, W, cam, rigid, xs, ys, bg_depth, n_fg, centroid, ws);     // odd background point, or none
}

// D of a multi-object edit: edit_points_splat_kernel with the point's object transform
__global__ void __launch_bounds__(256) edit_points_splat_objects_kernel(
    const float* __restrict__ bg_depth, int P, int H, int W, int K, CamDev cam, const dh_rigid* __restrict__ rigid,
    const float* __restrict__ xs, const float* __restrict__ ys, const int32_t* __restrict__ n_fg, const uint8_t* __restrict__ fg_object,
    const float* __restrict__ centroid, EditWs ws, int32_t* __restrict__ pix, uint64_t* __restrict__ zkey, double* __restrict__ dbg_points,
    uint64_t* zbuf) {
    const int e = blockIdx.y;
    const int n = n_fg[e] + ws.odd_count[e];
    uint64_t* zb = zbuf + (size_t)e * P;
    for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const int slot = base + threadIdx.x;
        const EditPoint pt = edit_point_objects(e, slot, P, W, K, cam, rigid, xs, ys, bg_depth, n_fg, fg_object, centroid, ws);
        int q = -1;
        uint64_t key = kEmptyZ;
        if (pt.live) {
            int u, v;
            const bool ok = project(cam, pt.X, pt.Y, pt.Z, H, W, u, v, key);
            q = ok ? v * W + u : -1;
            const size_t po = (size_t)e * 2 * P + pt.index;
            pix[po] = q; zkey[po] = key;
            if (dbg_points) {
                double* o = dbg_points + po * 3;
                o[0] = pt.X; o[1] = pt.Y; o[2] = pt.Z;
            }
        }
        zbuf_atomic_min_warp(zb, q, key);
    }
}

__global__ void __launch_bounds__(256) project_points_kernel(const double* __restrict__ points, int N, int H, int W,
                                                             CamDev cam, int32_t* __restrict__ pix, uint64_t* __restrict__ zkey,
                                                             int32_t* __restrict__ uo, int32_t* __restrict__ vo) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    int u, v;
    uint64_t key;
    const bool ok = project(cam, points[3 * (size_t)i], points[3 * (size_t)i + 1], points[3 * (size_t)i + 2], H, W, u, v, key);
    pix[i] = ok ? v * W + u : -1;
    zkey[i] = key;
    if (uo) uo[i] = u;
    if (vo) vo[i] = v;
}

// ------------------------------------------------------------------------------------------------
// transform_points (torch fp32 variant, depth_transform.py:439-459): centroid = mean over ALL points.
// Pairwise (deterministic) fp32 reduction; parity with torch is tolerance based.
// ------------------------------------------------------------------------------------------------
// block `blk` of `nblocks` (256 threads each, grid stride nblocks * 256) -> partial[3 blk .. 3 blk + 2]
__device__ __forceinline__ void tp_partial_sum(const float* __restrict__ pts, int N, int blk, int nblocks, double* __restrict__ partial) {
    __shared__ double sm[3][8];
    double s[3] = {0, 0, 0};
    for (int i = blk * blockDim.x + threadIdx.x; i < N; i += nblocks * blockDim.x) {
        s[0] += pts[3 * (size_t)i]; s[1] += pts[3 * (size_t)i + 1]; s[2] += pts[3 * (size_t)i + 2];
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[c] += __shfl_down_sync(0xFFFFFFFFu, s[c], o);
        if (lane_id() == 0) sm[c][warp_id()] = s[c];
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0;
        for (int w = 0; w < 8; ++w) t += sm[threadIdx.x][w];
        partial[blk * 3 + threadIdx.x] = t;
    }
}

__global__ void __launch_bounds__(256) tp_partial_sum_kernel(const float* __restrict__ pts, int N, double* __restrict__ partial) {
    tp_partial_sum(pts, N, blockIdx.x, gridDim.x, partial);
}

// the partial sums of every scene's foreground (blockIdx.y = scene), each with its own block count
__global__ void __launch_bounds__(256) tp_partial_sum_scenes_kernel(const float* __restrict__ pts, const SceneDesc* __restrict__ scenes,
                                                                    double* __restrict__ partial) {
    const SceneDesc sc = scenes[blockIdx.y];
    if ((int)blockIdx.x >= sc.tp_blocks) return;
    tp_partial_sum(pts + 3 * (size_t)sc.fg_v0, sc.V_fg, blockIdx.x, sc.tp_blocks, partial + 3 * (size_t)sc.tp_partial0);
}

// the centroid from the partial sums (every block repeats the short sum), then one point of one transform
__device__ __forceinline__ void tp_centroid(const double* __restrict__ partial, int nblocks, int N, float* cen) {
    if (threadIdx.x < 3) {
        double t = 0;
        for (int b = 0; b < nblocks; ++b) t += partial[b * 3 + threadIdx.x];
        cen[threadIdx.x] = (float)(t / (double)N);
    }
    __syncthreads();
}

__device__ __forceinline__ void tp_apply_point(const float* __restrict__ pts, int i, const float* cen, const TpEdit& e,
                                               float* __restrict__ out) {
    const float ax = e.ax, ay = e.ay, az = e.az, c = e.c, s = e.s;
    const float qx = pts[3 * (size_t)i] - cen[0], qy = pts[3 * (size_t)i + 1] - cen[1], qz = pts[3 * (size_t)i + 2] - cen[2];
    const float crx = ay * qz - az * qy, cry = az * qx - ax * qz, crz = ax * qy - ay * qx;
    const float d = qx * ax + qy * ay + qz * az;
    const float omc = 1.0f - c;
    out[3 * (size_t)i + 0] = (qx * c + crx * s + ax * d * omc) + cen[0] + e.tx;
    out[3 * (size_t)i + 1] = (qy * c + cry * s + ay * d * omc) + cen[1] + e.ty;
    out[3 * (size_t)i + 2] = (qz * c + crz * s + az * d * omc) + cen[2] + e.tz;
}

__global__ void __launch_bounds__(256) tp_apply_kernel(const float* __restrict__ pts, int N, const double* __restrict__ partial,
                                                       int nblocks, TpEdit e, float* __restrict__ out) {
    __shared__ float cen[3];
    tp_centroid(partial, nblocks, N, cen);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    tp_apply_point(pts, i, cen, e, out);
}

// B transforms of the same points: blockIdx.y = transform, output plane b = out + 3 N b
__global__ void __launch_bounds__(256) tp_apply_batch_kernel(const float* __restrict__ pts, int N, const double* __restrict__ partial,
                                                             int nblocks, const TpEdit* __restrict__ edits, float* __restrict__ out) {
    __shared__ float cen[3];
    tp_centroid(partial, nblocks, N, cen);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    const int b = blockIdx.y;
    tp_apply_point(pts, i, cen, edits[b], out + 3 * (size_t)N * b);
}

// edit b of a scene batch (blockIdx.y = edit): its scene's foreground moved with that scene's centroid
__global__ void __launch_bounds__(256) tp_apply_scenes_kernel(const float* __restrict__ pts, const SceneDesc* __restrict__ scenes,
                                                              const double* __restrict__ partial, const SceneEdit* __restrict__ edits,
                                                              float* __restrict__ out) {
    __shared__ float cen[3];
    const SceneEdit e = edits[blockIdx.y];
    const SceneDesc sc = scenes[e.scene];
    if ((int)(blockIdx.x * blockDim.x) >= sc.V_fg) return;          // uniform over the block, before the barrier
    tp_centroid(partial + 3 * (size_t)sc.tp_partial0, sc.tp_blocks, sc.V_fg, cen);
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= sc.V_fg) return;
    tp_apply_point(pts + 3 * (size_t)sc.fg_v0, i, cen, e.t, out + 3 * (size_t)e.out0);
}

int tp_partial_blocks(int N) { return N >= 256 * kTpMaxPartials ? kTpMaxPartials : (N + 255) / 256; }

int tp_transform_batch(const float* pts, int N, int B, const TpEdit* edits_dev, double* partial, float* out, cudaStream_t st) {
    const int nblocks = tp_partial_blocks(N);
    tp_partial_sum_kernel<<<nblocks, 256, 0, st>>>(pts, N, partial);
    DH_LAUNCH_CHECK();
    tp_apply_batch_kernel<<<dim3((N + 255) / 256, B), 256, 0, st>>>(pts, N, partial, nblocks, edits_dev, out);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int tp_transform_scenes(const float* pts, const SceneDesc* scenes_dev, int n_scenes, int max_blocks, const SceneEdit* edits_dev, int B,
                        int max_n, double* partial, float* out, cudaStream_t st) {
    if (max_n < 1) return DH_OK;
    tp_partial_sum_scenes_kernel<<<dim3(max_blocks, n_scenes), 256, 0, st>>>(pts, scenes_dev, partial);
    DH_LAUNCH_CHECK();
    tp_apply_scenes_kernel<<<dim3((max_n + 255) / 256, B), 256, 0, st>>>(pts, scenes_dev, partial, edits_dev, out);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

TpEdit tp_edit(float angle_degrees, const float* axis3, const float* translation3) {
    float a[3] = {axis3[0], axis3[1], axis3[2]};
    const float nrm = sqrtf(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
    for (float& v : a) v /= nrm;
    const float ang = angle_degrees * (float)(M_PI / 180.0);
    TpEdit e;
    e.ax = a[0]; e.ay = a[1]; e.az = a[2];
    e.c = cosf(ang); e.s = sinf(ang);
    e.tx = translation3[0]; e.ty = translation3[1]; e.tz = translation3[2];
    return e;
}

}  // namespace dh

using namespace dh;

extern "C" {

const char* dh_status_string(int status) {
    switch (status) {
        case DH_OK: return "ok";
        case DH_ERR_INVALID_ARGUMENT: return "invalid argument";
        case DH_ERR_UNSUPPORTED: return "unsupported";
        case DH_ERR_CUDA: return "CUDA runtime error";
        case DH_ERR_WORKSPACE: return "workspace too small";
        default: return "unknown status";
    }
}

int dh_abi_version(void) { return DH_B200_ABI_VERSION; }

int dh_last_cuda_error(void) { return g_last_cuda_error; }

int dh_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    DH_CUDA_CHECK(cudaGetDevice(&dev));
    if (sm_count) DH_CUDA_CHECK(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
    if (cc_major) DH_CUDA_CHECK(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    if (cc_minor) DH_CUDA_CHECK(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    return DH_OK;
}

int dh_linspace_f32_host(float start, float end, int steps, float* out) {
    DH_REQUIRE(out && steps >= 1);
    if (steps == 1) { out[0] = start; return DH_OK; }
    const float step = (end - start) / (float)(steps - 1);
    const int half = steps / 2;
    for (int i = 0; i < steps; ++i)
        out[i] = i < half ? fmaf(step, (float)i, start) : fmaf(-step, (float)(steps - 1 - i), end);
    return DH_OK;
}

int dh_unproject(const float* depth, int B, int H, int W, const dh_camera* cam_host, const float* xs, const float* ys,
                 float* points, void* stream) {
    DH_REQUIRE(depth && cam_host && xs && ys && points && B >= 1);
    DH_REQUIRE(H >= 2 && W >= 2);
    const int P = H * W;
    dim3 grid((P + 255) / 256, B);
    unproject_kernel<<<grid, 256, 0, as_stream(stream)>>>(depth, P, W, make_cam(cam_host), xs, ys, points);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

size_t dh_transform_points_workspace_bytes(int N) {
    (void)N;
    return kTpMaxPartials * 3 * sizeof(double);
}

int dh_transform_points(const float* points, int N, float angle_degrees, const float* axis_host3,
                        const float* translation_host3, float* out, void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(points && out && axis_host3 && translation_host3 && ws && N >= 1);
    if (ws_bytes < dh_transform_points_workspace_bytes(N)) return DH_ERR_WORKSPACE;
    const int nblocks = tp_partial_blocks(N);
    tp_partial_sum_kernel<<<nblocks, 256, 0, as_stream(stream)>>>(points, N, (double*)ws);
    DH_LAUNCH_CHECK();
    tp_apply_kernel<<<(N + 255) / 256, 256, 0, as_stream(stream)>>>(points, N, (const double*)ws, nblocks,
                                                                     tp_edit(angle_degrees, axis_host3, translation_host3), out);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

// workspace of the edit fast path behind the K1 layout: [odd_list int32 B*P][odd_count int32 B][minmax keys uint32 B*4]
struct EditWsOffsets { size_t odd_list, odd_count, minmax, total; };
static EditWsOffsets edit_ws_layout(int B, int P, size_t k1_bytes) {
    EditWsOffsets L;
    size_t o = k1_bytes;
    L.odd_list = o;  o = align_up(o + sizeof(int32_t) * (size_t)B * P, 256);
    L.odd_count = o; o = align_up(o + sizeof(int32_t) * (size_t)B, 256);
    L.minmax = o;    o = align_up(o + sizeof(uint32_t) * (size_t)B * 4, 256);
    L.total = o;
    return L;
}

// workspace of the fused pc path: [tile_counts int32 B*ntiles][rigid B][fgX][fgY][fgZ float B*P each]
static size_t k1_ws_layout(int B, int P, size_t* off_counts, size_t* off_rigid, size_t* off_x, size_t* off_y, size_t* off_z) {
    const int ntiles = (P + kTile - 1) / kTile;
    size_t o = 0;
    *off_counts = o; o = align_up(o + sizeof(int32_t) * (size_t)B * ntiles, 256);
    *off_rigid = o;  o = align_up(o + sizeof(dh_rigid) * (size_t)B, 256);
    *off_x = o;      o = align_up(o + sizeof(float) * (size_t)B * P, 256);
    *off_y = o;      o = align_up(o + sizeof(float) * (size_t)B * P, 256);
    *off_z = o;      o = align_up(o + sizeof(float) * (size_t)B * P, 256);
    return o;
}

size_t dh_edit_workspace_bytes(int B, int H, int W) {
    if (B < 1 || H < 1 || W < 1) return 0;
    size_t a, b, c, d, e;
    return edit_ws_layout(B, H * W, k1_ws_layout(B, H * W, &a, &b, &c, &d, &e)).total;
}

int dh_edit_splat(const float* depth, const float* bg_depth, const float* fg_mask, int B, int H, int W, const dh_camera* cam_host,
                  const dh_rigid* rigid_host, const float* xs, const float* ys, int32_t* pix, uint64_t* zkey, int32_t* fg_index,
                  int32_t* n_fg, float* centroid, double* points_out, uint64_t* zbuf, uint32_t* winner, float* depth_map,
                  uint8_t* target_mask, uint32_t* target_bits, int32_t* winner_src, float* inv_minmax, void* ws, size_t ws_bytes,
                  void* stream) {
    DH_REQUIRE(depth && bg_depth && fg_mask && cam_host && rigid_host && xs && ys && pix && zkey && fg_index && n_fg && centroid && ws);
    DH_REQUIRE(zbuf && winner && depth_map && target_bits);
    DH_REQUIRE(B >= 1 && H >= 2 && W >= 2);
    DH_REQUIRE((long long)H * W <= (1ll << 29));
    const int P = H * W;
    size_t oc, orr, ox, oy, oz;
    const size_t k1 = k1_ws_layout(B, P, &oc, &orr, &ox, &oy, &oz);
    const EditWsOffsets L = edit_ws_layout(B, P, k1);
    if (ws_bytes < L.total) return DH_ERR_WORKSPACE;
    char* w = static_cast<char*>(ws);
    EditWs ew;
    ew.tile_counts = reinterpret_cast<int32_t*>(w + oc);
    ew.rigid = reinterpret_cast<dh_rigid*>(w + orr);
    ew.fgX = reinterpret_cast<float*>(w + ox);
    ew.fgY = reinterpret_cast<float*>(w + oy);
    ew.fgZ = reinterpret_cast<float*>(w + oz);
    ew.odd_list = reinterpret_cast<int32_t*>(w + L.odd_list);
    ew.odd_count = reinterpret_cast<int32_t*>(w + L.odd_count);
    ew.minmax_keys = reinterpret_cast<uint32_t*>(w + L.minmax);
    cudaStream_t st = as_stream(stream);
    const CamDev cam = make_cam(cam_host);
    // the class for which a background point provably keeps its pixel: diagonal pinhole with K^-1 = 1/K (to fp32 rounding),
    // unit third row, square image (the x / y grids are linspace(-1, 1, S), engine.pixel_grid)
    const bool cam_nice = cam.diag && H == W && cam.k[8] == 1.0f && cam.kinv[8] == 1.0f && cam.k[0] > 0.0f && cam.k[4] > 0.0f &&
                          fabsf(cam.k[0] * cam.kinv[0] - 1.0f) < 1e-5f && fabsf(cam.k[4] * cam.kinv[4] - 1.0f) < 1e-5f && H <= 16384;
    const int ntiles = (P + kTile - 1) / kTile;
    const int wpr = (W + 31) / 32;
    DH_CUDA_CHECK(cudaMemcpyAsync(ew.rigid, rigid_host, sizeof(dh_rigid) * (size_t)B, cudaMemcpyHostToDevice, st));
    DH_CUDA_CHECK(cudaMemsetAsync(ew.odd_count, 0, sizeof(int32_t) * (size_t)B, st));
    dim3 tgrid(ntiles, B);
    edit_prepare_kernel<<<tgrid, kTileThreads, 0, st>>>(fg_mask, bg_depth, P, W, H, ntiles, cam_nice ? 1 : 0, cam, xs, ys, ew.tile_counts,
                                                        zbuf, ew, points_out ? pix : nullptr, points_out ? zkey : nullptr, points_out);
    DH_LAUNCH_CHECK();
    fg_compact_kernel<<<tgrid, kTileThreads, 0, st>>>(depth, fg_mask, P, W, ntiles, cam, xs, ys, ew.tile_counts, fg_index, ew.fgX, ew.fgY,
                                                      ew.fgZ, n_fg, nullptr);
    DH_LAUNCH_CHECK();
    fg_centroid_kernel<<<B, 96, 0, st>>>(ew.fgX, ew.fgY, ew.fgZ, n_fg, P, centroid);
    DH_LAUNCH_CHECK();
    // generic points (foreground + odd background): their number is only known on the device -> block-stride loops over a grid
    // that fills the GPU for any batch size (8 blocks of 256 per SM in total, at least 8 and at most 2 P / 256 per edit)
    int sms = 148;
    {
        int dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    int gx = (8 * sms + B - 1) / B;
    if (gx < 8) gx = 8;
    if (gx > (2 * P + 255) / 256) gx = (2 * P + 255) / 256;
    dim3 ggrid(gx, B);
    edit_points_splat_kernel<<<ggrid, 256, 0, st>>>(bg_depth, P, H, W, cam, ew.rigid, xs, ys, n_fg, centroid, ew, pix, zkey, points_out, zbuf);
    DH_LAUNCH_CHECK();
    int gr = (16 * sms + B - 1) / B;            // block-stride over the 32-pixel words of an edit
    if (gr < 16) gr = 16;
    if (gr > (H * wpr + 7) / 8) gr = (H * wpr + 7) / 8;
    edit_resolve_kernel<<<dim3(gr, B), 256, 0, st>>>(zbuf, bg_depth, H, W, wpr, cam_nice ? 1 : 0, winner, depth_map, target_mask,
                                                                   target_bits, winner_src, ew);
    DH_LAUNCH_CHECK();
    edit_points_winner_kernel<<<ggrid, 256, 0, st>>>(pix, zkey, n_fg, P, zbuf, winner, ew);
    DH_LAUNCH_CHECK();
    edit_points_publish_kernel<<<ggrid, 256, 0, st>>>(pix, n_fg, fg_index, P, W, wpr, winner, winner_src, target_mask, target_bits, ew,
                                                      inv_minmax);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

// workspace of a multi-object edit: the dh_edit_splat layout, then [tile_hist int32 B*ntiles*16][rigid B*16]
// [objX][objY][objZ float B*stride each]; stride holds the union plus 3 alignment floats per object
struct ObjWsOffsets { size_t tile_hist, rigid, x, y, z, stride, total; };
static ObjWsOffsets objects_ws_layout(int B, int P, size_t edit_bytes) {
    ObjWsOffsets L;
    const int ntiles = (P + kTile - 1) / kTile;
    L.stride = align_up((size_t)P + 4 * kMaxObjects, 64);
    size_t o = edit_bytes;
    L.tile_hist = o; o = align_up(o + sizeof(int32_t) * (size_t)B * ntiles * kMaxObjects, 256);
    L.rigid = o;     o = align_up(o + sizeof(dh_rigid) * (size_t)B * kMaxObjects, 256);
    L.x = o;         o = align_up(o + sizeof(float) * (size_t)B * L.stride, 256);
    L.y = o;         o = align_up(o + sizeof(float) * (size_t)B * L.stride, 256);
    L.z = o;         o = align_up(o + sizeof(float) * (size_t)B * L.stride, 256);
    L.total = o;
    return L;
}

size_t dh_edit_objects_workspace_bytes(int B, int H, int W) {
    if (B < 1 || H < 1 || W < 1) return 0;
    return objects_ws_layout(B, H * W, dh_edit_workspace_bytes(B, H, W)).total;
}

int dh_edit_splat_objects(const float* depth, const float* bg_depth, const float* fg_mask, const uint8_t* labels, int B, int K, int H,
                          int W, const dh_camera* cam_host, const dh_rigid* rigid_host, const float* xs, const float* ys, int32_t* pix,
                          uint64_t* zkey, int32_t* fg_index, uint8_t* fg_object, int32_t* n_fg, float* centroid, double* points_out,
                          uint64_t* zbuf, uint32_t* winner, float* depth_map, uint8_t* target_mask, uint32_t* target_bits,
                          int32_t* winner_src, float* inv_minmax, void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(depth && bg_depth && fg_mask && labels && cam_host && rigid_host && xs && ys && pix && zkey && fg_index && fg_object &&
               n_fg && centroid && ws);
    DH_REQUIRE(zbuf && winner && depth_map && target_bits);
    DH_REQUIRE(B >= 1 && H >= 2 && W >= 2 && K >= 1 && K <= kMaxObjects);
    DH_REQUIRE((long long)H * W <= (1ll << 29));
    const int P = H * W;
    size_t oc, orr, ox, oy, oz;
    const size_t k1 = k1_ws_layout(B, P, &oc, &orr, &ox, &oy, &oz);
    const EditWsOffsets L = edit_ws_layout(B, P, k1);
    const ObjWsOffsets O = objects_ws_layout(B, P, L.total);
    if (ws_bytes < O.total) return DH_ERR_WORKSPACE;
    char* w = static_cast<char*>(ws);
    EditWs ew;
    ew.tile_counts = reinterpret_cast<int32_t*>(w + oc);
    ew.rigid = reinterpret_cast<dh_rigid*>(w + O.rigid);          // [B][K]
    ew.fgX = reinterpret_cast<float*>(w + ox);
    ew.fgY = reinterpret_cast<float*>(w + oy);
    ew.fgZ = reinterpret_cast<float*>(w + oz);
    ew.odd_list = reinterpret_cast<int32_t*>(w + L.odd_list);
    ew.odd_count = reinterpret_cast<int32_t*>(w + L.odd_count);
    ew.minmax_keys = reinterpret_cast<uint32_t*>(w + L.minmax);
    ObjWs ow;
    ow.tile_hist = reinterpret_cast<int32_t*>(w + O.tile_hist);
    ow.objX = reinterpret_cast<float*>(w + O.x);
    ow.objY = reinterpret_cast<float*>(w + O.y);
    ow.objZ = reinterpret_cast<float*>(w + O.z);
    ow.stride = O.stride;
    cudaStream_t st = as_stream(stream);
    const CamDev cam = make_cam(cam_host);
    // the camera / image class of dh_edit_splat in which a background point provably keeps its pixel
    const bool cam_nice = cam.diag && H == W && cam.k[8] == 1.0f && cam.kinv[8] == 1.0f && cam.k[0] > 0.0f && cam.k[4] > 0.0f &&
                          fabsf(cam.k[0] * cam.kinv[0] - 1.0f) < 1e-5f && fabsf(cam.k[4] * cam.kinv[4] - 1.0f) < 1e-5f && H <= 16384;
    const int ntiles = (P + kTile - 1) / kTile;
    const int wpr = (W + 31) / 32;
    DH_CUDA_CHECK(cudaMemcpyAsync(ew.rigid, rigid_host, sizeof(dh_rigid) * (size_t)B * K, cudaMemcpyHostToDevice, st));
    DH_CUDA_CHECK(cudaMemsetAsync(ew.odd_count, 0, sizeof(int32_t) * (size_t)B, st));
    dim3 tgrid(ntiles, B);
    edit_prepare_kernel<<<tgrid, kTileThreads, 0, st>>>(fg_mask, bg_depth, P, W, H, ntiles, cam_nice ? 1 : 0, cam, xs, ys, ew.tile_counts,
                                                        zbuf, ew, points_out ? pix : nullptr, points_out ? zkey : nullptr, points_out);
    DH_LAUNCH_CHECK();
    fg_compact_objects_kernel<<<tgrid, kTileThreads, 0, st>>>(depth, fg_mask, labels, P, W, ntiles, K, cam, xs, ys, ew.tile_counts, fg_index,
                                                              fg_object, ew.fgX, ew.fgY, ew.fgZ, n_fg, ow.tile_hist);
    DH_LAUNCH_CHECK();
    fg_centroid_objects_kernel<<<dim3(K, B), 256, 0, st>>>(ew.fgX, ew.fgY, ew.fgZ, fg_object, n_fg, P, ntiles, K, ow, centroid);
    DH_LAUNCH_CHECK();
    // the grids of dh_edit_splat
    int sms = 148;
    {
        int dev = 0;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    int gx = (8 * sms + B - 1) / B;
    if (gx < 8) gx = 8;
    if (gx > (2 * P + 255) / 256) gx = (2 * P + 255) / 256;
    dim3 ggrid(gx, B);
    edit_points_splat_objects_kernel<<<ggrid, 256, 0, st>>>(bg_depth, P, H, W, K, cam, ew.rigid, xs, ys, n_fg, fg_object, centroid, ew, pix,
                                                           zkey, points_out, zbuf);
    DH_LAUNCH_CHECK();
    int gr = (16 * sms + B - 1) / B;
    if (gr < 16) gr = 16;
    if (gr > (H * wpr + 7) / 8) gr = (H * wpr + 7) / 8;
    edit_resolve_kernel<<<dim3(gr, B), 256, 0, st>>>(zbuf, bg_depth, H, W, wpr, cam_nice ? 1 : 0, winner, depth_map, target_mask,
                                                                   target_bits, winner_src, ew);
    DH_LAUNCH_CHECK();
    edit_points_winner_kernel<<<ggrid, 256, 0, st>>>(pix, zkey, n_fg, P, zbuf, winner, ew);
    DH_LAUNCH_CHECK();
    edit_points_publish_kernel<<<ggrid, 256, 0, st>>>(pix, n_fg, fg_index, P, W, wpr, winner, winner_src, target_mask, target_bits, ew,
                                                      inv_minmax);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_transform_point_cloud(const float* points, const float* mask, int N, const dh_rigid* rigid_host, double* out,
                             float* centroid, int32_t* n_masked, void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(points && mask && rigid_host && out && centroid && n_masked && ws && N >= 1);
    // workspace = the K1 layout for one "image" of N pixels (+ the compacted index list)
    size_t oc, orr, ox, oy, oz;
    const size_t k1 = k1_ws_layout(1, N, &oc, &orr, &ox, &oy, &oz);
    if (ws_bytes < k1 + sizeof(int32_t) * (size_t)N) return DH_ERR_WORKSPACE;
    char* w = static_cast<char*>(ws);
    int32_t* tile_counts = reinterpret_cast<int32_t*>(w + oc);
    dh_rigid* rigid_dev = reinterpret_cast<dh_rigid*>(w + orr);
    float* fgX = reinterpret_cast<float*>(w + ox);
    float* fgY = reinterpret_cast<float*>(w + oy);
    float* fgZ = reinterpret_cast<float*>(w + oz);
    int32_t* index = reinterpret_cast<int32_t*>(w + k1);
    cudaStream_t st = as_stream(stream);
    const int ntiles = (N + kTile - 1) / kTile;
    CamDev cam;
    memset(&cam, 0, sizeof(cam));
    DH_CUDA_CHECK(cudaMemcpyAsync(rigid_dev, rigid_host, sizeof(dh_rigid), cudaMemcpyHostToDevice, st));
    fg_count_kernel<<<dim3(ntiles, 1), kTileThreads, 0, st>>>(mask, N, ntiles, tile_counts);
    DH_LAUNCH_CHECK();
    fg_compact_kernel<<<dim3(ntiles, 1), kTileThreads, 0, st>>>(nullptr, mask, N, N, ntiles, cam, nullptr, nullptr, tile_counts, index,
                                                               fgX, fgY, fgZ, n_masked, points);
    DH_LAUNCH_CHECK();
    fg_centroid_kernel<<<1, 96, 0, st>>>(fgX, fgY, fgZ, n_masked, N, centroid);
    DH_LAUNCH_CHECK();
    rigid_all_kernel<<<(N + 255) / 256, 256, 0, st>>>(points, N, rigid_dev, centroid, out);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

size_t dh_transform_point_cloud_workspace_bytes(int N) {
    if (N < 1) return 0;
    size_t a, b, c, d, e;
    return k1_ws_layout(1, N, &a, &b, &c, &d, &e) + sizeof(int32_t) * (size_t)N;
}

int dh_project_points(const double* points, int N, int H, int W, const dh_camera* cam_host, int32_t* pix, uint64_t* zkey,
                      int32_t* u, int32_t* v, void* stream) {
    DH_REQUIRE(points && cam_host && pix && zkey && N >= 0 && H >= 1 && W >= 1);
    if (N == 0) return DH_OK;
    project_points_kernel<<<(N + 255) / 256, 256, 0, as_stream(stream)>>>(points, N, H, W, make_cam(cam_host), pix, zkey, u, v);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // extern "C"
