// Shared device/host helpers of libdiffhandles_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>

#include "../../include/dh_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libdiffhandles_b200 is written for sm_100a (B200) only"
#endif

namespace dh {

extern thread_local int g_last_cuda_error;

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = static_cast<int>(e);
    return DH_ERR_CUDA;
}

#define DH_CUDA_CHECK(expr)                                   \
    do {                                                      \
        cudaError_t _e = (expr);                              \
        if (_e != cudaSuccess) return ::dh::cuda_fail(_e);    \
    } while (0)

#define DH_LAUNCH_CHECK() DH_CUDA_CHECK(cudaPeekAtLastError())

#define DH_REQUIRE(cond)                                      \
    do {                                                      \
        if (!(cond)) return DH_ERR_INVALID_ARGUMENT;          \
    } while (0)

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

constexpr uint32_t kNoWinner = 0xFFFFFFFFu;
constexpr uint64_t kEmptyZ = 0xFFFFFFFFFFFFFFFFull;

// Order-preserving map fp64 -> uint64 (negative values sort below positive ones; -0 is folded into +0
// by the caller).  Inverse below.
__host__ __device__ inline uint64_t z_to_key(double z) {
#ifdef __CUDA_ARCH__
    uint64_t b = static_cast<uint64_t>(__double_as_longlong(z));
#else
    uint64_t b;
    memcpy(&b, &z, 8);
#endif
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}

__device__ inline double key_to_z(uint64_t k) {
    uint64_t b = (k & 0x8000000000000000ull) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k;
    return __longlong_as_double(static_cast<long long>(b));
}

// Order-preserving map fp32 -> uint32 for atomicMin/atomicMax on floats.
__device__ inline uint32_t f_to_key(float f) {
    uint32_t b = __float_as_uint(f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ inline float key_to_f(uint32_t k) {
    uint32_t b = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
    return __uint_as_float(b);
}

// transform_points (dh_geometry.cu) for B rigid transforms of one point set: the constants of one transform, prepared on the
// host as dh_transform_points prepares them, and the launcher that applies B of them in one pass.  Transform b writes
// out[3 N b .. 3 N (b + 1)), bit-identical to dh_transform_points with that transform.  `partial` holds 3 * kTpMaxPartials
// doubles.
constexpr int kTpMaxPartials = 256;
struct TpEdit {
    float ax, ay, az;    // unit rotation axis
    float c, s;          // cos / sin of the angle
    float tx, ty, tz;    // translation
};
TpEdit tp_edit(float angle_degrees, const float* axis3, const float* translation3);
int tp_transform_batch(const float* pts, int N, int B, const TpEdit* edits_dev, double* partial, float* out, cudaStream_t st);

// One scene of a scene table (device copy; offsets into concatenated per-scene arrays) and one edit of a scene batch.
// tp_transform_scenes moves the V_fg foreground points of edit b's scene (pts + 3 fg_v0) by its transform into
// out + 3 out0 with the centroid of that scene alone, bit-identical to dh_transform_points on that scene: each scene sums its
// partials with its own block count and stride (tp_partial_blocks of its V_fg) into partial + 3 tp_partial0.
struct SceneDesc {
    int bg_v0, V_bg, bg_f0, F_bg;    // background vertices / faces (faces scene-local)
    int fg_v0, V_fg, fg_f0, F_fg;    // foreground vertices (and colours) / faces (faces scene-local)
    int tp_blocks, tp_partial0;      // centroid partial sums of the foreground
    int plane;                       // the edit whose key plane receives the background raster (-1: no edit uses the scene)
};
struct SceneEdit {
    TpEdit t;
    int scene;
    int out0;                        // first moved vertex of this edit in the flat (sum over edits of V_fg) arrays
};
int tp_partial_blocks(int N);
int tp_transform_scenes(const float* pts, const SceneDesc* scenes_dev, int n_scenes, int max_blocks, const SceneEdit* edits_dev, int B,
                        int max_n, double* partial, float* out, cudaStream_t st);

__device__ inline int warp_id() { return threadIdx.x >> 5; }
__device__ inline int lane_id() { return threadIdx.x & 31; }

// Pass 1 of the z-buffer splat for one point per lane (q < 0: no point), called by all 32 lanes: zb[q] = min(zb[q], key).
// When every lane hits one pixel - clamped off-screen points pile onto border pixels - the warp reduces its keys (high halves,
// then the low halves of the lanes that hold the minimal high half) and issues one atomic.  A plain load first shows whether
// the key can win at all: the buffer only ever decreases, so a stale read is conservative.
__device__ __forceinline__ void zbuf_atomic_min_warp(uint64_t* zb, int q, uint64_t key) {
    const unsigned full = 0xFFFFFFFFu;
    const int q0 = __shfl_sync(full, q, 0);
    if (__all_sync(full, q == q0)) {
        if (q0 < 0) return;
        const uint32_t hi = (uint32_t)(key >> 32), lo = (uint32_t)key;
        const uint32_t mhi = __reduce_min_sync(full, hi);
        const uint32_t mlo = __reduce_min_sync(full, hi == mhi ? lo : 0xFFFFFFFFu);
        if (lane_id() == 0) {
            const uint64_t m = ((uint64_t)mhi << 32) | mlo;
            if (m < *(volatile uint64_t*)(zb + q0)) atomicMin((unsigned long long*)(zb + q0), (unsigned long long)m);
        }
        return;
    }
    if (q >= 0 && key < *(volatile uint64_t*)(zb + q)) atomicMin((unsigned long long*)(zb + q), (unsigned long long)key);
}

// Exclusive scan of one int per thread over a CTA of up to 1024 threads; returns the exclusive prefix,
// writes the CTA total to `total`.  `smem` needs 33 ints.
__device__ inline int block_exclusive_scan(int v, int* smem, int& total) {
    const int lane = lane_id(), wid = warp_id();
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int n = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= o) inc += n;
    }
    if (lane == 31) smem[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        int nw = (blockDim.x + 31) >> 5;
        int w = lane < nw ? smem[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int n = __shfl_up_sync(0xFFFFFFFFu, winc, o);
            if (lane >= o) winc += n;
        }
        smem[lane] = winc - w;
        if (lane == 31) smem[32] = winc;
    }
    __syncthreads();
    int res = smem[wid] + inc - v;
    total = smem[32];
    __syncthreads();
    return res;
}

}  // namespace dh
