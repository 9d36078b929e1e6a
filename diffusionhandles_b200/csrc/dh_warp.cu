// K3: the activation warp (SURVEY.md 8(a) row 9) - winner-index gather over NCHW fp32 activation stacks.
//
// Dense form: out[e][c][q] = map[e][q] >= 0 ? in[e][c][map[e][q]] : 0 for every level of a stack.
// HBM-bound permutation copy: algorithmic bytes = read source once + write destination once (+ maps).
//
// Fast path (every named SD2-depth shape: 64^2x320, 32^2x640, 16^2x1280, 8^2x1280 and the recorded
// 32^2x1280 / 64^2x640 / 64^2x320 stacks): a persistent, warp-specialised kernel.
//   * the source planes of one (edit, level) are contiguous, so they are cut into 16 KB chunks
//     (1 plane of 64^2, 4 of 32^2, 16 of 16^2, 64 of 8^2); one producer thread streams the chunks into a
//     ring of shared-memory stages with TMA bulk copies (cp.async.bulk.shared::cluster.global +
//     mbarrier complete_tx; SASS: UBLKCP) - no registers, no LSU on the global-load side;
//   * 8 consumer warps gather from shared memory through per-thread offsets that are computed ONCE per
//     segment (the map is the same for every channel of a level) and kept in 16 registers, and write
//     the destination with 128-bit streaming stores, fully coalesced (512 B per warp instruction);
//   * full/empty mbarriers per stage; the producer runs ahead across segment boundaries.
// Generic path: any (C, hw, n) - direct global gather with int4 index loads and float4 stores; also the
// list form W[c][n] = A[c][idx[n]] that the reference losses consume (losses.py:46-47, :80).
#include "dh_common.cuh"
#include "dh_tma.cuh"

#include <stdlib.h>
#include <string.h>

namespace dh {

constexpr int kStageFloats = 4096;                 // 16 KB
constexpr int kStageBytes = kStageFloats * 4;
constexpr int kConsumerThreads = 256;
constexpr int kWarpThreads = kConsumerThreads + 32;
constexpr int kSlotsPerThread = kStageFloats / 4 / kConsumerThreads;   // float4 slots per thread per stage = 4
constexpr int kMaxLevels = 8;

struct LevelDev {
    const float* in;
    float* out;
    const int32_t* map;
    int hw;                // cells per plane
    int edit_floats;       // C * hw
    int chunks_per_edit;   // ceil(edit_floats / kStageFloats)
    int seg_chunks;        // chunks per segment
    int segs_per_edit;
    int seg_begin;         // first global segment id of this level
};

struct WarpParams {
    LevelDev lv[kMaxLevels];
    int n_levels;
    int total_segs;
};

__device__ __forceinline__ void st_stream_f4(float* p, float4 v) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

struct Segment {
    int level, edit, c0, c1;
};

__device__ __forceinline__ Segment decode_segment(const WarpParams& p, int seg) {
    int l = 0;
#pragma unroll
    for (int i = 1; i < kMaxLevels; ++i)
        if (i < p.n_levels && seg >= p.lv[i].seg_begin) l = i;
    const LevelDev& L = p.lv[l];
    const int local = seg - L.seg_begin;
    Segment s;
    s.level = l;
    s.edit = local / L.segs_per_edit;
    const int si = local - s.edit * L.segs_per_edit;
    s.c0 = si * L.seg_chunks;
    s.c1 = min(L.chunks_per_edit, s.c0 + L.seg_chunks);
    return s;
}

template <int kStages>
__global__ void __launch_bounds__(kWarpThreads) warp_dense_tma_kernel(const __grid_constant__ WarpParams p) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    float* stages = reinterpret_cast<float*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)kStages * kStageBytes);
    uint64_t* empty = full + kStages;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) {
            mbar_init(full + s, 1);
            mbar_init(empty + s, kConsumerThreads / 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (threadIdx.x >= kConsumerThreads) {
        // ===== producer warp: one elected lane streams chunks into the stage ring =====
        if (threadIdx.x == kConsumerThreads) {
            uint32_t stage = 0, phase = 0;
            for (int seg = blockIdx.x; seg < p.total_segs; seg += gridDim.x) {
                const Segment sg = decode_segment(p, seg);
                const LevelDev& L = p.lv[sg.level];
                const float* src = L.in + (size_t)sg.edit * L.edit_floats;
                for (int c = sg.c0; c < sg.c1; ++c) {
                    mbar_wait(empty + stage, phase ^ 1);
                    const int floats = min(kStageFloats, L.edit_floats - c * kStageFloats);
                    mbar_arrive_expect_tx(full + stage, (uint32_t)floats * 4u);
                    tma_bulk_g2s(stages + (size_t)stage * kStageFloats, src + (size_t)c * kStageFloats, (uint32_t)floats * 4u, full + stage);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
        return;
    }

    // ===== consumers =====
    const int t = threadIdx.x;
    uint32_t stage = 0, phase = 0;
    for (int seg = blockIdx.x; seg < p.total_segs; seg += gridDim.x) {
        const Segment sg = decode_segment(p, seg);
        const LevelDev& L = p.lv[sg.level];
        const int hw = L.hw;
        const int32_t* map = L.map + (size_t)sg.edit * hw;
        // per-thread gather offsets inside a stage; identical for every chunk of the level because a stage
        // holds a whole number of planes
        int off[kSlotsPerThread][4];
#pragma unroll
        for (int k = 0; k < kSlotsPerThread; ++k) {
            const int el = 4 * (t + kConsumerThreads * k);
            const int plane = el / hw;
            const int q0 = el - plane * hw;
            const int4 m = *reinterpret_cast<const int4*>(map + q0);
            // (unsigned compare: negative = "no source", and an index >= hw from a caller's own map is treated the same way
            // instead of reading outside the stage)
            off[k][0] = (unsigned)m.x < (unsigned)hw ? plane * hw + m.x : -1;
            off[k][1] = (unsigned)m.y < (unsigned)hw ? plane * hw + m.y : -1;
            off[k][2] = (unsigned)m.z < (unsigned)hw ? plane * hw + m.z : -1;
            off[k][3] = (unsigned)m.w < (unsigned)hw ? plane * hw + m.w : -1;
        }
        float* dst = L.out + (size_t)sg.edit * L.edit_floats;
        for (int c = sg.c0; c < sg.c1; ++c) {
            const int floats = min(kStageFloats, L.edit_floats - c * kStageFloats);
            mbar_wait(full + stage, phase);
            const float* sm = stages + (size_t)stage * kStageFloats;
            float4 v[kSlotsPerThread];
#pragma unroll
            for (int k = 0; k < kSlotsPerThread; ++k) {
                v[k].x = off[k][0] >= 0 ? sm[off[k][0]] : 0.0f;
                v[k].y = off[k][1] >= 0 ? sm[off[k][1]] : 0.0f;
                v[k].z = off[k][2] >= 0 ? sm[off[k][2]] : 0.0f;
                v[k].w = off[k][3] >= 0 ? sm[off[k][3]] : 0.0f;
            }
            float* o = dst + (size_t)c * kStageFloats;
#pragma unroll
            for (int k = 0; k < kSlotsPerThread; ++k) {
                const int el = 4 * (t + kConsumerThreads * k);
                if (el < floats) st_stream_f4(o + el, v[k]);
            }
            // hand the stage back to the producer only after the stores: a store cannot issue before the shared loads
            // it reads have returned, while the mbarrier arrive does not wait for loads still in flight - arriving
            // right after the loads let the next TMA copy overwrite the stage under a few late loads
            __syncwarp();
            if ((t & 31) == 0) mbar_arrive(empty + stage);
            if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
    }
}

// ---- generic gather: out[c][i] = idx[i] >= 0 ? in[c][idx[i]] : 0 ------------------------------------
constexpr int kGenChannels = 8;

// out_aligned: `out` is 16-byte aligned.  Only then (and with n % 4 == 0) is every row group a float4 slot; a caller's
// view at an odd float offset takes the scalar stores.
__global__ void __launch_bounds__(256) gather_generic_kernel(const float* __restrict__ in, int C, int hw_in,
                                                             const int32_t* __restrict__ idx, int n, float* __restrict__ out,
                                                             int out_aligned) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;       // group of 4 consecutive outputs
    const int i0 = g * 4;
    if (i0 >= n) return;
    const int c0 = blockIdx.y * kGenChannels;
    const int c1 = min(C, c0 + kGenChannels);
    const bool vec = out_aligned && (i0 + 3 < n) && ((n & 3) == 0);
    int id[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) id[j] = (i0 + j < n) ? idx[i0 + j] : -1;
    for (int c = c0; c < c1; ++c) {
        const float* a = in + (size_t)c * hw_in;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) v[j] = (unsigned)id[j] < (unsigned)hw_in ? __ldg(a + id[j]) : 0.0f;   // out of range -> 0, never a wild read
        float* o = out + (size_t)c * n + i0;
        if (vec) {
            *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j < n) o[j] = v[j];
        }
    }
}

}  // namespace dh

using namespace dh;

namespace {

constexpr int kStagesDefault = 4;
constexpr int kCtasPerSmDefault = 1;
constexpr int kSegChunksDefault = 10;

int sm_count_cached() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
    }
    return sms;
}

bool fast_path_ok(const dh_warp_level& l) {
    if (l.hw <= 0 || l.hw > kStageFloats || (kStageFloats % l.hw) != 0 || (l.hw % 4) != 0) return false;
    if ((reinterpret_cast<uintptr_t>(l.in) & 15) || (reinterpret_cast<uintptr_t>(l.out) & 15) ||
        (reinterpret_cast<uintptr_t>(l.src_map) & 15))
        return false;
    return (((size_t)l.channels * l.hw) % 4) == 0;
}

}  // namespace

template <int kStages>
static int launch_dense(const WarpParams& p, int ctas_per_sm, cudaStream_t st) {
    const size_t smem = (size_t)kStages * kStageBytes + 2 * kStages * sizeof(uint64_t);
    DH_CUDA_CHECK(cudaFuncSetAttribute(warp_dense_tma_kernel<kStages>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int grid = sm_count_cached() * ctas_per_sm;
    if (grid > p.total_segs) grid = p.total_segs;
    warp_dense_tma_kernel<kStages><<<grid, kWarpThreads, smem, st>>>(p);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

extern "C" {

int dh_warp_gather_list(const float* in, int C, int hw, const int32_t* idx, int n, float* out, void* stream) {
    DH_REQUIRE(in && out && C >= 1 && hw >= 1 && n >= 0 && (idx || n == 0));
    if (n == 0) return DH_OK;
    dim3 grid(((n + 3) / 4 + 255) / 256, (C + kGenChannels - 1) / kGenChannels);
    const int out_aligned = (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    gather_generic_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, C, hw, idx, n, out, out_aligned);
    DH_LAUNCH_CHECK();
    return DH_OK;
}

// Tunables (environment): DH_WARP_STAGES (2,3,4,6,8), DH_WARP_CTAS_PER_SM, DH_WARP_SEG_CHUNKS.
int dh_warp_gather_dense(const dh_warp_level* levels_host, int n_levels, int B, void* stream) {
    DH_REQUIRE(levels_host && n_levels >= 1 && n_levels <= kMaxLevels && B >= 1);
    cudaStream_t st = as_stream(stream);
    const char* ea = getenv("DH_WARP_CTAS_PER_SM");
    const char* eb = getenv("DH_WARP_SEG_CHUNKS");
    const char* ec = getenv("DH_WARP_STAGES");
    int stages = ec ? atoi(ec) : kStagesDefault;
    int ctas_per_sm = ea ? atoi(ea) : kCtasPerSmDefault;
    int seg_chunks_cfg = eb ? atoi(eb) : kSegChunksDefault;
    if (ctas_per_sm < 1 || ctas_per_sm > 8) ctas_per_sm = kCtasPerSmDefault;
    if (seg_chunks_cfg < 1) seg_chunks_cfg = kSegChunksDefault;
    // every level is checked before the first launch: a rejected call writes no output
    for (int i = 0; i < n_levels; ++i) {
        const dh_warp_level& l = levels_host[i];
        DH_REQUIRE(l.in && l.out && l.src_map && l.channels >= 1 && l.hw >= 1 && l.in != l.out);
    }
    WarpParams p;
    memset(&p, 0, sizeof(p));
    int nfast = 0, seg = 0;
    for (int i = 0; i < n_levels; ++i) {
        const dh_warp_level& l = levels_host[i];
        if (!fast_path_ok(l)) {
            // generic path, one launch per edit
            for (int e = 0; e < B; ++e) {
                int rc = dh_warp_gather_list(l.in + (size_t)e * l.channels * l.hw, l.channels, l.hw, l.src_map + (size_t)e * l.hw,
                                             l.hw, l.out + (size_t)e * l.channels * l.hw, stream);
                if (rc) return rc;
            }
            continue;
        }
        LevelDev& L = p.lv[nfast++];
        L.in = l.in; L.out = l.out; L.map = l.src_map;
        L.hw = l.hw;
        L.edit_floats = l.channels * l.hw;
        L.chunks_per_edit = (L.edit_floats + kStageFloats - 1) / kStageFloats;
        L.seg_chunks = seg_chunks_cfg < L.chunks_per_edit ? seg_chunks_cfg : L.chunks_per_edit;
        L.segs_per_edit = (L.chunks_per_edit + L.seg_chunks - 1) / L.seg_chunks;
        L.seg_begin = seg;
        seg += L.segs_per_edit * B;
    }
    if (nfast == 0) return DH_OK;
    p.n_levels = nfast;
    p.total_segs = seg;
    switch (stages) {
        case 2: return launch_dense<2>(p, ctas_per_sm, st);
        case 3: return launch_dense<3>(p, ctas_per_sm, st);
        case 6: return launch_dense<6>(p, ctas_per_sm, st);
        case 8: return launch_dense<8>(p, ctas_per_sm, st);
        default: return launch_dense<4>(p, ctas_per_sm, st);
    }
}

}  // extern "C"
