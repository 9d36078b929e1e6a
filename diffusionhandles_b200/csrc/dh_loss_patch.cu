// K4, general patch size: local-average guidance losses with patch_size > 1 (losses.py:51-84, SURVEY.md 8(f) rank 4).
//
// The reference replaces both maps by their local averages over the indexed cells before taking the L1 difference:
//     F[c,q] = (box_p(w * up)[c,q] / p^2) / (box_p(w)[q] / p^2 + 1e-10),    w = 1 on the indexed cells,
// box_p = the window sum of AvgPool2d(p, stride 1, padding p//2) (zero padded, divisor always p^2), and autograd sends
// the gradient back through the average of the current map.  Every shipped configuration uses p = 1 (dh_loss.cu);
// this kernel serves the general case with the same plan (dh_build_loss_plan), the same layer descriptors and the same
// loss_out layout, so the host side only switches the entry point.
//
// One CTA per SM walks over (layer, channel) planes.  Everything of one plane lives in shared memory at the loss-grid
// resolution (ten 16 KB planes at 64 x 64): the two resized maps, their local averages, an INTEGER plane that
// accumulates the sign terms of the pairs (associative -> the gradient is bit-reproducible), and the gradient, which is
// brought back through the transposed box filter and the transposed bilinear resize in gather form (no float atomics).
// The per-channel loss terms go to a partial array that a one-CTA kernel reduces in a fixed order.
//
// dh_guidance_loss_patch_batch runs up to 16 edits in one launch: every CTA serves one edit with that edit's parameters and
// partial array, and the finish kernel reduces each edit in its own CTA, so every edit gets the bits of its own launch.
#include "dh_common.cuh"
#include "dh_loss_plan.cuh"

#include <string.h>

#include "../../include/dh_b200.h"

namespace dh {

constexpr int kPatchThreads = 512;
constexpr int kPatchWarps = kPatchThreads / 32;
constexpr int kMaxPatch = 31;

struct PatchLayer {
    const float* cur;
    const float* orig;
    float* grad;
    int C, h, w;
    float fgw, bgw;
    int chan_begin;
};

struct PatchParams {
    PatchLayer lv[kMaxLossLayers];
    int n_layers, total_channels, G, patch;
    const void* plan;
    int plan_cap;
    int n_fg, n_bg_orig, n_bg_trans, n_bg_common;
    int fg_kind, bg_kind;
    float* partial;     // [total_channels][2]: fg sum, bg term
    float* loss_out;
};

__device__ __forceinline__ float patch_block_sum(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    __syncthreads();                                  // the previous result has been consumed
    if (lane_id() == 0) red[warp_id()] = v;
    __syncthreads();
    float t = lane_id() < kPatchWarps ? red[lane_id()] : 0.0f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xFFFFFFFFu, t, o);
    return t;
}

// out[y][x] = sum_{d in [0,p)} in[y][x + off + d] (zero outside), optionally masked on the input side
template <bool kMasked>
__device__ __forceinline__ void hbox(const float* __restrict__ in, const unsigned char* __restrict__ flags, unsigned bit,
                                     float* __restrict__ out, int G, int p, int off) {
    for (int q = threadIdx.x; q < G * G; q += kPatchThreads) {
        const int y = q / G, x = q - y * G;
        const int a = max(0, x + off), b = min(G - 1, x + off + p - 1);
        float s = 0.0f;
        for (int j = a; j <= b; ++j) {
            const float v = in[y * G + j];
            s += kMasked ? ((flags[y * G + j] & bit) ? v : 0.0f) : v;
        }
        out[q] = s;
    }
}

__device__ __forceinline__ float vbox_at(const float* __restrict__ in, int G, int p, int off, int y, int x) {
    const int a = max(0, y + off), b = min(G - 1, y + off + p - 1);
    float s = 0.0f;
    for (int j = a; j <= b; ++j) s += in[j * G + x];
    return s;
}

// One local-average L1 term (foreground pairs, or the background list paired with itself).  On return `gu` has
// received the gradient w.r.t. the resized current map and the CTA-wide sum of mult * |difference| is returned.
template <bool kBackground>
__device__ float local_term(const PatchParams& p, const PlanView& pv, const float* __restrict__ u1, const float* __restrict__ u2,
                            float* __restrict__ f1, float* __restrict__ f2, float* __restrict__ tmp, int* __restrict__ gi,
                            float* __restrict__ gu, const float* __restrict__ den1, const float* __restrict__ den2,
                            const unsigned char* __restrict__ flags, float scale, float* red) {
    const int G = p.G, cells = G * G, P = p.patch, pad = P / 2;
    const float pp = (float)(P * P);
    const unsigned bit1 = kBackground ? 4u : 1u, bit2 = kBackground ? 4u : 2u;
    const int tid = threadIdx.x;
    hbox<true>(u1, flags, bit1, tmp, G, P, -pad);
    __syncthreads();
    for (int q = tid; q < cells; q += kPatchThreads) f1[q] = vbox_at(tmp, G, P, -pad, q / G, q % G) / pp / den1[q];
    __syncthreads();
    hbox<true>(u2, flags, bit2, tmp, G, P, -pad);
    for (int q = tid; q < cells; q += kPatchThreads) gi[q] = 0;
    __syncthreads();
    for (int q = tid; q < cells; q += kPatchThreads) f2[q] = vbox_at(tmp, G, P, -pad, q / G, q % G) / pp / den2[q];
    __syncthreads();
    float acc = 0.0f;
    if (kBackground) {
        for (int q = tid; q < cells; q += kPatchThreads) {
            const int m = pv.bgcnt[q].z;
            if (m == 0) continue;
            const float d = f1[q] - f2[q];
            acc += (float)m * fabsf(d);
            gi[q] = d > 0.0f ? -m : (d < 0.0f ? m : 0);
        }
    } else {
        const int n_pairs = pv.row_ptr[cells];
        for (int k = tid; k < n_pairs; k += kPatchThreads) {
            const uint2 e = pv.pairs[k];
            const int s = (int)(e.x & 0xFFFFu), d = (int)(e.x >> 16), m = (int)e.y;
            const float df = f1[s] - f2[d];
            acc += (float)m * fabsf(df);
            if (df != 0.0f) atomicAdd(gi + d, df > 0.0f ? -m : m);
        }
    }
    acc = patch_block_sum(acc, red);                    // contains barriers: gi is complete afterwards
    // back through the average: dL/dA2[q] = g[q] / den2[q]; A2 = box(w2 * u2) / p^2
    for (int q = tid; q < cells; q += kPatchThreads) f1[q] = scale * (float)gi[q] / den2[q] / pp;
    __syncthreads();
    // transposed window: cell j is inside the windows of q in [j + pad - P + 1, j + pad]
    hbox<false>(f1, flags, 0u, tmp, G, P, pad - P + 1);
    __syncthreads();
    for (int q = tid; q < cells; q += kPatchThreads)
        if (flags[q] & bit2) gu[q] += vbox_at(tmp, G, P, pad - P + 1, q / G, q % G);
    __syncthreads();
    return acc;
}

// The work of CTA cta.index() of the cta.count() CTAs that serve one edit: the edit's weight maps and denominators, then the
// planes index, index + count, ...  A plane's partial and gradient do not depend on which CTA computes them.
template <class Cta>
__device__ __forceinline__ void loss_patch_body(const PatchParams& p, Cta cta) {
    extern __shared__ __align__(16) float psm[];
    __shared__ float red[kPatchWarps];
    __shared__ int tap0[2][kMaxG], tap1[2][kMaxG];       // [0] rows, [1] columns of the current layer
    __shared__ float lam[2][kMaxG];
    __shared__ int win_lo[2][kMaxNative], win_hi[2][kMaxNative];
    const int G = p.G, cells = G * G, tid = threadIdx.x;
    float* const u1 = psm;
    float* const u2 = u1 + cells;
    float* const tmp = u2 + cells;
    float* const f1 = tmp + cells;
    float* const f2 = f1 + cells;
    float* const gu = f2 + cells;
    int* const gi = reinterpret_cast<int*>(gu + cells);
    float* const den_f1 = reinterpret_cast<float*>(gi + cells);
    float* const den_f2 = den_f1 + cells;
    float* const den_b = den_f2 + cells;
    unsigned char* const flags = reinterpret_cast<unsigned char*>(den_b + cells);
    PlanView pv = plan_view(const_cast<void*>(p.plan), G, p.plan_cap);
    const int P = p.patch, pad = P / 2;
    const float pp = (float)(P * P);

    // ---- once per CTA: the weight maps of the three lists and the denominators box(w) / p^2 + 1e-10 ----
    for (int q = tid; q < cells; q += kPatchThreads) {
        const ushort4 bc = pv.bgcnt[q];
        flags[q] = (unsigned char)((bc.w & 1u) | (pv.row_ptr[q + 1] > pv.row_ptr[q] ? 2u : 0u) | (bc.z > 0 ? 4u : 0u));
    }
    __syncthreads();
    for (int which = 0; which < 3; ++which) {
        float* den = which == 0 ? den_f1 : (which == 1 ? den_f2 : den_b);
        const unsigned bit = 1u << which;
        for (int q = tid; q < cells; q += kPatchThreads) u1[q] = (flags[q] & bit) ? 1.0f : 0.0f;
        __syncthreads();
        hbox<false>(u1, flags, 0u, tmp, G, P, -pad);
        __syncthreads();
        for (int q = tid; q < cells; q += kPatchThreads) den[q] = vbox_at(tmp, G, P, -pad, q / G, q % G) / pp + 1e-10f;
        __syncthreads();
    }

    int cur_layer = -1;
    for (int gc = cta.index(); gc < p.total_channels; gc += cta.count()) {
        int l = 0;
        for (int i = 1; i < p.n_layers; ++i)
            if (gc >= p.lv[i].chan_begin) l = i;
        const PatchLayer& L = p.lv[l];
        const int c = gc - L.chan_begin, h = L.h, w = L.w;
        const bool native = h == G && w == G;
        const float* __restrict__ vc = L.cur + (size_t)c * h * w;
        const float* __restrict__ vo = L.orig + (size_t)c * h * w;
        if (!native && l != cur_layer) {
            // bilinear taps of this layer and, per native row / column, the range of up rows / columns that tap it
            __syncthreads();
            for (int i = tid; i < 2 * G; i += kPatchThreads) {
                const int ax = i / G, k = i - ax * G, n = ax == 0 ? h : w;
                int a, b; float t;
                bilinear_tap(k, n, (float)n / (float)G, a, b, t);
                tap0[ax][k] = a; tap1[ax][k] = b; lam[ax][k] = t;
            }
            __syncthreads();
            for (int i = tid; i < h + w; i += kPatchThreads) {
                const int ax = i < h ? 0 : 1, k = ax == 0 ? i : i - h;
                int lo = G, hi = -1;
                for (int j = 0; j < G; ++j)
                    if (tap0[ax][j] == k || tap1[ax][j] == k) { lo = min(lo, j); hi = max(hi, j); }
                win_lo[ax][k] = lo; win_hi[ax][k] = hi;
            }
            __syncthreads();
        }
        cur_layer = l;

        // ---- the two maps at the loss-grid resolution ----
        if (native) {
            // 128-bit accesses only when the planes and the shared-memory maps are 16-byte aligned: with a cell count that is not a
            // multiple of four, plane c >= 1 and the map u2 (at psm + cells) start at offsets that are not
            const bool vec = (cells & 3) == 0 && ((reinterpret_cast<uintptr_t>(vc) | reinterpret_cast<uintptr_t>(vo)) & 15) == 0;
            const int n4 = vec ? cells / 4 : 0;
            for (int q = tid; q < n4; q += kPatchThreads) {
                reinterpret_cast<float4*>(u2)[q] = __ldg(reinterpret_cast<const float4*>(vc) + q);
                reinterpret_cast<float4*>(u1)[q] = __ldg(reinterpret_cast<const float4*>(vo) + q);
            }
            for (int q = n4 * 4 + tid; q < cells; q += kPatchThreads) { u2[q] = vc[q]; u1[q] = vo[q]; }
        } else {
            for (int q = tid; q < cells; q += kPatchThreads) {
                const int Y = q / G, X = q - Y * G;
                const int y0 = tap0[0][Y], y1 = tap1[0][Y], x0 = tap0[1][X], x1 = tap1[1][X];
                const float ly = lam[0][Y], lx = lam[1][X];
                const float c00 = __ldg(vc + y0 * w + x0), c01 = __ldg(vc + y0 * w + x1), c10 = __ldg(vc + y1 * w + x0), c11 = __ldg(vc + y1 * w + x1);
                const float o00 = __ldg(vo + y0 * w + x0), o01 = __ldg(vo + y0 * w + x1), o10 = __ldg(vo + y1 * w + x0), o11 = __ldg(vo + y1 * w + x1);
                u2[q] = (1.0f - ly) * ((1.0f - lx) * c00 + lx * c01) + ly * ((1.0f - lx) * c10 + lx * c11);
                u1[q] = (1.0f - ly) * ((1.0f - lx) * o00 + lx * o01) + ly * ((1.0f - lx) * o10 + lx * o11);
            }
        }
        for (int q = tid; q < cells; q += kPatchThreads) gu[q] = 0.0f;
        __syncthreads();

        float fg_sum = 0.0f, bg_term = 0.0f;
        if (p.fg_kind) {
            const float scale = p.n_fg > 0 ? L.fgw / ((float)L.C * (float)p.n_fg) : 0.0f;
            fg_sum = local_term<false>(p, pv, u1, u2, f1, f2, tmp, gi, gu, den_f1, den_f2, flags, scale, red);
        }
        if (p.bg_kind == 2) {
            const float scale = p.n_bg_common > 0 ? L.bgw / ((float)L.C * (float)p.n_bg_common) : 0.0f;
            bg_term = local_term<true>(p, pv, u1, u2, f1, f2, tmp, gi, gu, den_b, den_b, flags, scale, red);
        } else if (p.bg_kind == 1) {
            float s1 = 0.0f, s2 = 0.0f;
            for (int q = tid; q < cells; q += kPatchThreads) {
                const ushort4 bc = pv.bgcnt[q];
                s1 += (float)bc.x * u1[q];
                s2 += (float)bc.y * u2[q];
            }
            s1 = patch_block_sum(s1, red);
            s2 = patch_block_sum(s2, red);
            const float delta = s1 / (float)p.n_bg_orig - s2 / (float)p.n_bg_trans;
            bg_term = fabsf(delta);
            const float gscale = p.n_bg_trans > 0 ? L.bgw / ((float)L.C * (float)p.n_bg_trans) : 0.0f;
            const float gval = -sgn(delta) * gscale;
            for (int q = tid; q < cells; q += kPatchThreads) gu[q] += gval * (float)pv.bgcnt[q].y;
            __syncthreads();
        }
        if (tid == 0) { p.partial[2 * gc] = fg_sum; p.partial[2 * gc + 1] = bg_term; }

        // ---- gradient at native resolution ----
        if (L.grad) {
            float* __restrict__ g = L.grad + (size_t)c * h * w;
            if (native) {
                for (int q = tid; q < cells; q += kPatchThreads) g[q] = gu[q];
            } else {
                // transposed bilinear resize, gather form: columns first (tmp[Y][x]), then rows
                for (int i = tid; i < G * w; i += kPatchThreads) {
                    const int Y = i / w, x = i - Y * w;
                    float s = 0.0f;
                    for (int X = win_lo[1][x]; X <= win_hi[1][x]; ++X) {
                        const float t = lam[1][X];
                        const float cf = (tap0[1][X] == x ? 1.0f - t : 0.0f) + (tap1[1][X] == x ? t : 0.0f);
                        s += cf * gu[Y * G + X];
                    }
                    tmp[i] = s;
                }
                __syncthreads();
                for (int i = tid; i < h * w; i += kPatchThreads) {
                    const int y = i / w, x = i - y * w;
                    float s = 0.0f;
                    for (int Y = win_lo[0][y]; Y <= win_hi[0][y]; ++Y) {
                        const float t = lam[0][Y];
                        const float cf = (tap0[0][Y] == y ? 1.0f - t : 0.0f) + (tap1[0][Y] == y ? t : 0.0f);
                        s += cf * tmp[Y * w + x];
                    }
                    g[i] = s;
                }
            }
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kPatchThreads, 1) loss_patch_kernel(const __grid_constant__ PatchParams p) {
    loss_patch_body(p, WholeGrid{});
}

// Several edits in one launch: CTAs [cta_begin[e], cta_begin[e + 1]) serve edit e exactly as a loss_patch_kernel launch of
// that many CTAs would.  Every edit writes its own partial array and gradients; grid and patch are launch-wide.
struct PatchBatchParams {
    PatchParams edit[kMaxBatchEdits];
    int cta_begin[kMaxBatchEdits + 1];
    int n_edits;
};
static_assert(sizeof(PatchBatchParams) <= 32764, "kernel parameters are limited to 32764 bytes");

struct EditCtas {
    int first, n;       // first CTA of the edit, CTAs of the edit
    __device__ __forceinline__ int index() const { return (int)blockIdx.x - first; }
    __device__ __forceinline__ int count() const { return n; }
};

__global__ void __launch_bounds__(kPatchThreads, 1) loss_patch_batch_kernel(const __grid_constant__ PatchBatchParams bp) {
    int e = 0;
#pragma unroll
    for (int i = 1; i < kMaxBatchEdits; ++i)
        if (i < bp.n_edits && (int)blockIdx.x >= bp.cta_begin[i]) e = i;
    loss_patch_body(bp.edit[e], EditCtas{bp.cta_begin[e], bp.cta_begin[e + 1] - bp.cta_begin[e]});
}

// fixed-order reduction of the per-channel terms: loss_out[0] = total, [1+2l] = fg_l, [2+2l] = bg_l
__device__ __forceinline__ void loss_patch_finish(const PatchParams& p) {
    __shared__ float red[kPatchWarps];
    float total = 0.0f;
    for (int l = 0; l < p.n_layers; ++l) {
        const PatchLayer& L = p.lv[l];
        float a = 0.0f, b = 0.0f;
        for (int c = threadIdx.x; c < L.C; c += kPatchThreads) {
            a += p.partial[2 * (L.chan_begin + c)];
            b += p.partial[2 * (L.chan_begin + c) + 1];
        }
        a = patch_block_sum(a, red);
        b = patch_block_sum(b, red);
        const float fg = p.fg_kind ? a / (float)p.n_fg / (float)L.C : 0.0f;
        const float bg = p.bg_kind == 2 ? b / (float)p.n_bg_common / (float)L.C : (p.bg_kind == 1 ? b / (float)L.C : 0.0f);
        if (threadIdx.x == 0) { p.loss_out[1 + 2 * l] = fg; p.loss_out[2 + 2 * l] = bg; }
        if (p.fg_kind) total += L.fgw * fg;
        if (p.bg_kind) total += L.bgw * bg;
    }
    if (threadIdx.x == 0) p.loss_out[0] = total;
}

__global__ void __launch_bounds__(kPatchThreads) loss_patch_finish_kernel(const __grid_constant__ PatchParams p) {
    loss_patch_finish(p);
}

// one CTA per edit, each the single-edit reduction of that edit
__global__ void __launch_bounds__(kPatchThreads) loss_patch_finish_batch_kernel(const __grid_constant__ PatchBatchParams bp) {
    loss_patch_finish(bp.edit[blockIdx.x]);
}

static size_t patch_smem_bytes(int grid) {
    const size_t cells = (size_t)grid * grid;
    return cells * 10 * sizeof(float) + ((cells + 15) / 16) * 16;
}

// Validates one edit and builds its PatchParams, with its partial array at the start of ws.  No CUDA call.
static int prepare_patch_edit(const dh_loss_layer* layers_host, int n_layers, int grid, int patch_size, const void* plan, int n_fg,
                              int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind, float* loss_out, void* ws,
                              size_t ws_bytes, PatchParams& p) {
    DH_REQUIRE(layers_host && plan && loss_out && ws);
    DH_REQUIRE(n_layers >= 1 && n_layers <= kMaxLossLayers && grid >= 1 && grid <= kMaxG);
    DH_REQUIRE(patch_size >= 1 && patch_size <= kMaxPatch);
    DH_REQUIRE(n_fg >= 0 && n_bg_orig >= 0 && n_bg_trans >= 0 && n_bg_common >= 0);
    DH_REQUIRE(fg_kind >= 0 && fg_kind <= 1 && bg_kind >= 0 && bg_kind <= 2);
    memset(&p, 0, sizeof(p));
    int total = 0;
    for (int l = 0; l < n_layers; ++l) {
        const dh_loss_layer& s = layers_host[l];
        DH_REQUIRE(s.cur && s.orig && s.channels >= 1 && s.h >= 1 && s.w >= 1 && s.h <= grid && s.w <= grid);
        DH_REQUIRE(s.h <= kMaxNative && s.w <= kMaxNative);
        PatchLayer& d = p.lv[l];
        d.cur = s.cur; d.orig = s.orig; d.grad = s.grad; d.C = s.channels; d.h = s.h; d.w = s.w;
        d.fgw = s.fg_weight; d.bgw = s.bg_weight; d.chan_begin = total;
        total += s.channels;
    }
    if (ws_bytes < (size_t)total * 2 * sizeof(float)) return DH_ERR_WORKSPACE;
    p.n_layers = n_layers; p.total_channels = total; p.G = grid; p.patch = patch_size;
    p.plan = plan; p.plan_cap = n_fg;
    p.n_fg = n_fg; p.n_bg_orig = n_bg_orig; p.n_bg_trans = n_bg_trans; p.n_bg_common = n_bg_common;
    p.fg_kind = fg_kind; p.bg_kind = bg_kind;
    p.partial = static_cast<float*>(ws); p.loss_out = loss_out;
    return DH_OK;
}

static int sm_count(int* sms) {
    int dev = 0;
    DH_CUDA_CHECK(cudaGetDevice(&dev));
    DH_CUDA_CHECK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return DH_OK;
}

// one edit: min(channels, SMs) CTAs of loss_patch_kernel, then the one-CTA reduction
static int launch_patch_edit(const PatchParams& p, void* stream) {
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != DH_OK) return rc;
    const size_t smem = patch_smem_bytes(p.G);
    DH_CUDA_CHECK(cudaFuncSetAttribute(loss_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ctas = p.total_channels < sms ? p.total_channels : sms;
    loss_patch_kernel<<<ctas, kPatchThreads, smem, as_stream(stream)>>>(p);
    DH_LAUNCH_CHECK();
    loss_patch_finish_kernel<<<1, kPatchThreads, 0, as_stream(stream)>>>(p);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

// several edits of one grid: CTAs in proportion to the edits' channels, at least one per edit, none without a plane, and at
// most the SM count in all (each CTA holds a whole SM: 512 threads and up to 160 KB of shared memory)
static int launch_patch_batch(PatchBatchParams& bp, int n_edits, void* stream) {
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc != DH_OK) return rc;
    long long channels = 0;
    for (int e = 0; e < n_edits; ++e) channels += bp.edit[e].total_channels;
    const long long spare = sms > n_edits ? sms - n_edits : 0;
    int n_ctas = 0;
    for (int e = 0; e < n_edits; ++e) {
        const int c = bp.edit[e].total_channels;
        int share = 1 + (int)(spare * c / channels);
        if (share > c) share = c;
        bp.cta_begin[e] = n_ctas;
        n_ctas += share;
    }
    bp.cta_begin[n_edits] = n_ctas;
    bp.n_edits = n_edits;
    const size_t smem = patch_smem_bytes(bp.edit[0].G);
    DH_CUDA_CHECK(cudaFuncSetAttribute(loss_patch_batch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    loss_patch_batch_kernel<<<n_ctas, kPatchThreads, smem, as_stream(stream)>>>(bp);
    DH_LAUNCH_CHECK();
    loss_patch_finish_batch_kernel<<<n_edits, kPatchThreads, 0, as_stream(stream)>>>(bp);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

}  // namespace dh

using namespace dh;

extern "C" {

size_t dh_guidance_loss_patch_workspace_bytes(int n_layers, int max_channels) {
    if (n_layers < 1 || n_layers > kMaxLossLayers || max_channels < 1) return 0;
    return (size_t)n_layers * (size_t)max_channels * 2 * sizeof(float);
}

int dh_guidance_loss_patch(const dh_loss_layer* layers_host, int n_layers, int grid, int patch_size, const void* plan, int n_fg,
                           int n_bg_orig, int n_bg_trans, int n_bg_common, int fg_kind, int bg_kind, float* loss_out, void* ws,
                           size_t ws_bytes, void* stream) {
    PatchParams p;
    const int rc = prepare_patch_edit(layers_host, n_layers, grid, patch_size, plan, n_fg, n_bg_orig, n_bg_trans, n_bg_common, fg_kind,
                                      bg_kind, loss_out, ws, ws_bytes, p);
    return rc != DH_OK ? rc : launch_patch_edit(p, stream);
}

size_t dh_guidance_loss_patch_batch_workspace_bytes(int n_edits, int n_layers, int max_channels) {
    if (n_edits < 1 || n_edits > kMaxBatchEdits) return 0;
    return (size_t)n_edits * dh_guidance_loss_patch_workspace_bytes(n_layers, max_channels);
}

int dh_guidance_loss_patch_batch(const dh_loss_batch_edit* edits_host, int n_edits, int grid, int patch_size, int fg_kind, int bg_kind,
                                 void* ws, size_t ws_bytes, void* stream) {
    DH_REQUIRE(edits_host && ws && n_edits >= 1);
    if (n_edits > kMaxBatchEdits) return DH_ERR_UNSUPPORTED;
    PatchBatchParams bp;
    memset(&bp, 0, sizeof(bp));
    // edit e owns bytes [e * stride, (e + 1) * stride) of the workspace (a partial array is a multiple of 8 bytes)
    const size_t stride = ws_bytes / (size_t)n_edits / 8 * 8;
    for (int e = 0; e < n_edits; ++e) {
        const dh_loss_batch_edit& E = edits_host[e];
        const int rc = prepare_patch_edit(E.layers, E.n_layers, grid, patch_size, E.plan, E.n_fg, E.n_bg_orig, E.n_bg_trans, E.n_bg_common,
                                          fg_kind, bg_kind, E.loss_out, static_cast<char*>(ws) + e * stride, stride, bp.edit[e]);
        if (rc != DH_OK) return rc;
    }
    return n_edits == 1 ? launch_patch_edit(bp.edit[0], stream) : launch_patch_batch(bp, n_edits, stream);
}

}  // extern "C"
