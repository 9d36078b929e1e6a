// K2: deterministic z-buffered point splat (SURVEY.md 8(a) row 5) and its epilogue.
//
// The reference (depth_transform.py:697-712) visits the points in index order and replaces a pixel's
// depth on a strict '<', so the winner of pixel q is the lexicographic minimum of (z_i, i) over the
// points that land on q.  z is fp64 and i needs 20+ bits, so the pair does not fit one 64-bit atomic.
// It is resolved exactly with two passes:
//   pass 1: zbuf[q]   = atomicMin over order-preserving 64-bit keys of z_i           (ULL atomicMin)
//   pass 2: winner[q] = atomicMin over { i : key_i == zbuf[q] }                       (u32 atomicMin)
// Both passes pre-reduce inside a warp when all of its lanes hit the same pixel (clamped off-screen
// points pile onto border pixels by the tens of thousands, SURVEY.md config 5) and skip the atomic when
// a plain load already shows the point cannot win (the buffers only ever decrease, so a stale read is
// conservative).
#include "dh_common.cuh"

#include <cooperative_groups.h>

namespace dh {

__device__ __forceinline__ int edit_points(const int32_t* n_points, int n_fixed, int e) {
    return n_fixed + (n_points ? n_points[e] : 0);
}

__global__ void __launch_bounds__(256) splat_z_kernel(const int32_t* __restrict__ pix, const uint64_t* __restrict__ zkey,
                                                      const int32_t* __restrict__ n_points, int n_fixed, int stride, int P,
                                                      uint64_t* zbuf) {
    const int e = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = edit_points(n_points, n_fixed, e);
    int q = -1;
    uint64_t key = kEmptyZ;
    if (i < n) {
        q = pix[(size_t)e * stride + i];
        key = zkey[(size_t)e * stride + i];
    }
    zbuf_atomic_min_warp(zbuf + (size_t)e * P, q, key);
}

__global__ void __launch_bounds__(256) splat_winner_kernel(const int32_t* __restrict__ pix, const uint64_t* __restrict__ zkey,
                                                           const int32_t* __restrict__ n_points, int n_fixed, int stride, int P,
                                                           const uint64_t* __restrict__ zbuf, uint32_t* winner) {
    const int e = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = edit_points(n_points, n_fixed, e);
    int q = -1;
    bool tie = false;
    if (i < n) {
        q = pix[(size_t)e * stride + i];
        if (q >= 0) tie = zkey[(size_t)e * stride + i] == zbuf[(size_t)e * P + q];
    }
    uint32_t* wb = winner + (size_t)e * P;
    const unsigned full = 0xFFFFFFFFu;
    const int q0 = __shfl_sync(full, q, 0);
    if (__all_sync(full, q == q0)) {
        if (q0 < 0) return;
        const uint32_t m = __reduce_min_sync(full, tie ? (uint32_t)i : kNoWinner);
        if (lane_id() == 0 && m != kNoWinner && m < *(volatile uint32_t*)(wb + q0)) atomicMin(wb + q0, m);
        return;
    }
    if (tie && (uint32_t)i < *(volatile uint32_t*)(wb + q)) atomicMin(wb + q, (uint32_t)i);
}

// One warp per 32-pixel word of a row: writes depth_map / target_mask / winner_src and the packed mask.
__global__ void __launch_bounds__(256) splat_resolve_kernel(const uint64_t* __restrict__ zbuf, const uint32_t* __restrict__ winner,
                                                            int H, int W, int wpr, int fg_start, const uint8_t* __restrict__ point_mask,
                                                            const int32_t* __restrict__ fg_index, int stride,
                                                            float* __restrict__ depth_map, uint8_t* __restrict__ target_mask,
                                                            uint32_t* __restrict__ target_bits, int32_t* __restrict__ winner_src) {
    const int e = blockIdx.y;
    const int word = blockIdx.x * (blockDim.x >> 5) + warp_id();
    if (word >= H * wpr) return;
    const int row = word / wpr, col = (word - row * wpr) * 32 + lane_id();
    const int P = H * W;
    bool fg = false;
    if (col < W) {
        const size_t q = (size_t)e * P + row * W + col;
        const uint32_t w = winner[q];
        float d = __int_as_float(0x7F800000);   // +inf: empty pixel (depth_transform.py:689)
        int32_t src = -1;
        if (w != kNoWinner) {
            d = __double2float_rn(key_to_z(zbuf[q]));
            if (point_mask) {
                fg = point_mask[(size_t)e * stride + w] != 0;
                src = (int32_t)w;
            } else {
                fg = (int)w >= fg_start;
                src = fg ? (fg_index ? fg_index[(size_t)e * P + (w - fg_start)] : (int32_t)w) : (int32_t)w;
            }
        }
        if (depth_map) depth_map[q] = d;
        if (target_mask) target_mask[q] = fg ? 1 : 0;
        if (winner_src) winner_src[q] = src;
    }
    const uint32_t bits = __ballot_sync(0xFFFFFFFFu, fg);
    if (target_bits && lane_id() == 0) target_bits[(size_t)e * H * wpr + word] = bits;
}

__global__ void __launch_bounds__(256) splat_visible_kernel(const int32_t* __restrict__ pix, const uint32_t* __restrict__ winner,
                                                            const int32_t* __restrict__ n_points, int n_fixed, int stride, int P,
                                                            int fg_start, const uint8_t* __restrict__ point_mask,
                                                            uint8_t* __restrict__ visible) {
    const int e = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= edit_points(n_points, n_fixed, e)) return;
    const size_t pi = (size_t)e * stride + i;
    const int q = pix[pi];
    const bool fg = point_mask ? point_mask[pi] != 0 : i >= fg_start;
    visible[pi] = (fg && q >= 0 && winner[(size_t)e * P + q] == (uint32_t)i) ? 1 : 0;
}

// min / max of 1/depth over one image.  A thread-block CLUSTER of 8 CTAs works on one edit: every CTA reduces an
// eighth of the image into its own shared memory, then rank 0 reads the seven other partial results through
// distributed shared memory (no scratch buffer, no atomics, deterministic).  IEEE division is monotone, so instead of
// dividing every pixel the kernel tracks min/max of the non-negative and of the negative depths and takes four
// reciprocals at the end: bit-identical to min/max over fl(1/d).
constexpr int kMinMaxCluster = 8;

__global__ void __cluster_dims__(kMinMaxCluster, 1, 1) __launch_bounds__(512)
inv_minmax_kernel(const float* __restrict__ depth, int P, float* __restrict__ out) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ float sm[4][16];
    __shared__ float part[4];
    const int e = blockIdx.y;
    const unsigned rank = cluster.block_rank();
    const float* d = depth + (size_t)e * P;
    const float inf = __int_as_float(0x7F800000);
    float pmin = inf, pmax = -inf, nmin = inf, nmax = -inf;     // over sign-bit-clear / sign-bit-set values
    auto take = [&](float x) {
        if (x != x) return;
        if (__float_as_uint(x) & 0x80000000u) { nmin = fminf(nmin, x); nmax = fmaxf(nmax, x); }
        else { pmin = fminf(pmin, x); pmax = fmaxf(pmax, x); }
    };
    const int P4 = ((reinterpret_cast<uintptr_t>(d) & 15) == 0) ? P / 4 : 0;
    for (int i = rank * blockDim.x + threadIdx.x; i < P4; i += kMinMaxCluster * blockDim.x) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(d) + i);
        take(v.x); take(v.y); take(v.z); take(v.w);
    }
    for (int p = P4 * 4 + rank * blockDim.x + threadIdx.x; p < P; p += kMinMaxCluster * blockDim.x) take(d[p]);
    float r[4] = {pmin, -pmax, nmin, -nmax};                      // all four as minima
#pragma unroll
    for (int k = 0; k < 4; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r[k] = fminf(r[k], __shfl_xor_sync(0xFFFFFFFFu, r[k], o));
        if (lane_id() == 0) sm[k][warp_id()] = r[k];
    }
    __syncthreads();
    if (warp_id() == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            r[k] = lane_id() < (int)(blockDim.x >> 5) ? sm[k][lane_id()] : inf;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) r[k] = fminf(r[k], __shfl_xor_sync(0xFFFFFFFFu, r[k], o));
            if (lane_id() == 0) part[k] = r[k];
        }
    }
    cluster.sync();
    if (rank == 0 && threadIdx.x == 0) {
        float q[4] = {inf, inf, inf, inf};
        for (unsigned b = 0; b < kMinMaxCluster; ++b) {
            const float* rp = cluster.map_shared_rank(part, b);
#pragma unroll
            for (int k = 0; k < 4; ++k) q[k] = fminf(q[k], rp[k]);
        }
        pmin = q[0]; pmax = -q[1]; nmin = q[2]; nmax = -q[3];
        float mn = inf, mx = -inf;
        if (pmin <= pmax) {           // some non-negative depth: reciprocals in [1/pmax, 1/pmin]
            mn = fminf(mn, __fdiv_rn(1.0f, pmax));
            mx = fmaxf(mx, __fdiv_rn(1.0f, pmin));
        }
        if (nmin <= nmax) {           // some negative depth: reciprocals in [1/nmax, 1/nmin]
            mn = fminf(mn, __fdiv_rn(1.0f, nmax));
            mx = fmaxf(mx, __fdiv_rn(1.0f, nmin));
        }
        out[e * 2] = mn;
        out[e * 2 + 1] = mx;
    }
    cluster.sync();      // keep every CTA's shared memory alive until rank 0 has read it
}

// normalize_depth(1/depth): (255 * (x - min)) / (max - min), fp32, same operation order as the reference.
__global__ void __launch_bounds__(256) disparity_kernel(const float* __restrict__ depth, int P, const float* __restrict__ bounds,
                                                        float* __restrict__ disp) {
    const int e = blockIdx.y;
    const float mn = bounds[e * 2], mx = bounds[e * 2 + 1];
    const float range = __fsub_rn(mx, mn);
    const float* d = depth + (size_t)e * P;
    float* o = disp + (size_t)e * P;
    auto one = [&](float v) { return __fdiv_rn(__fmul_rn(255.0f, __fsub_rn(__fdiv_rn(1.0f, v), mn)), range); };
    const int p0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;       // four pixels per thread: 128-bit loads and stores
    if (p0 + 3 < P && ((((size_t)e * P) & 3) == 0) && ((reinterpret_cast<uintptr_t>(depth) | reinterpret_cast<uintptr_t>(disp)) & 15) == 0) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(d + p0));
        *reinterpret_cast<float4*>(o + p0) = make_float4(one(v.x), one(v.y), one(v.z), one(v.w));
    } else {
        for (int p = p0; p < min(P, p0 + 4); ++p) o[p] = one(d[p]);
    }
}

}  // namespace dh

using namespace dh;

extern "C" {

int dh_splat_zbuffer(const int32_t* pix, const uint64_t* zkey, const int32_t* n_points, int n_fixed, int n_max,
                     int stride_points, int B, int P, uint64_t* zbuf, uint32_t* winner, void* stream) {
    DH_REQUIRE(pix && zkey && zbuf && winner && B >= 1 && P >= 1 && n_max >= 0 && stride_points >= n_max);
    cudaStream_t st = as_stream(stream);
    DH_CUDA_CHECK(cudaMemsetAsync(zbuf, 0xFF, sizeof(uint64_t) * (size_t)B * P, st));
    DH_CUDA_CHECK(cudaMemsetAsync(winner, 0xFF, sizeof(uint32_t) * (size_t)B * P, st));
    if (n_max == 0) return DH_OK;
    dim3 grid((n_max + 255) / 256, B);
    splat_z_kernel<<<grid, 256, 0, st>>>(pix, zkey, n_points, n_fixed, stride_points, P, zbuf);
    DH_LAUNCH_CHECK();
    splat_winner_kernel<<<grid, 256, 0, st>>>(pix, zkey, n_points, n_fixed, stride_points, P, zbuf, winner);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_splat_resolve(const uint64_t* zbuf, const uint32_t* winner, int B, int H, int W, int fg_start,
                     const uint8_t* point_mask, const int32_t* fg_index, int stride_points, float* depth_map,
                     uint8_t* target_mask, uint32_t* target_bits, int32_t* winner_src, float* inv_minmax, void* stream) {
    DH_REQUIRE(zbuf && winner && B >= 1 && H >= 1 && W >= 1);
    cudaStream_t st = as_stream(stream);
    const int wpr = (W + 31) / 32;
    const int words = H * wpr;
    dim3 grid((words + 7) / 8, B);
    splat_resolve_kernel<<<grid, 256, 0, st>>>(zbuf, winner, H, W, wpr, fg_start, point_mask, fg_index, stride_points,
                                               depth_map, target_mask, target_bits, winner_src);
    DH_LAUNCH_CHECK();
    if (inv_minmax) {
        DH_REQUIRE(depth_map);
        inv_minmax_kernel<<<dim3(kMinMaxCluster, B), 512, 0, st>>>(depth_map, H * W, inv_minmax);
        DH_LAUNCH_CHECK();
    }
    return DH_OK;
}

int dh_splat_visible(const int32_t* pix, const uint32_t* winner, const int32_t* n_points, int n_fixed, int n_max,
                     int stride_points, int B, int P, int fg_start, const uint8_t* point_mask, uint8_t* visible, void* stream) {
    DH_REQUIRE(pix && winner && visible && B >= 1 && P >= 1 && n_max >= 0);
    if (n_max == 0) return DH_OK;
    dim3 grid((n_max + 255) / 256, B);
    splat_visible_kernel<<<grid, 256, 0, as_stream(stream)>>>(pix, winner, n_points, n_fixed, stride_points, P, fg_start,
                                                              point_mask, visible);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_inv_minmax(const float* depth, int B, int P, float* inv_minmax, void* stream) {
    DH_REQUIRE(depth && inv_minmax && B >= 1 && P >= 1);
    inv_minmax_kernel<<<dim3(kMinMaxCluster, B), 512, 0, as_stream(stream)>>>(depth, P, inv_minmax);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

int dh_disparity(const float* depth, int B, int P, const float* bounds, float* disparity, void* stream) {
    DH_REQUIRE(depth && bounds && disparity && B >= 1 && P >= 1);
    dim3 grid((P + 1023) / 1024, B);
    disparity_kernel<<<grid, 256, 0, as_stream(stream)>>>(depth, P, bounds, disparity);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // extern "C"
