// rt_sort.cuh -- inter-bounce ray reordering (the role of Ref::SortRays_CPU, reference internal/CoreRef.cpp:1667-1710,
// and of the GPU reference's 8-pass LSD radix sort, internal/RendererGPU.h:756-780).
//
// The step is results-neutral: every pixel owns at most one ray per bounce and each ray carries its pixel in `xy`, so
// the ORDER of the ray list never reaches the image (SURVEY.md section 8(a) row a13).  What matters is that rays that
// start close together and point the same way sit next to each other so a warp walks the same BVH nodes.  So instead of
// reproducing the reference's 32-bit hash + full radix sort (~240 B/ray), this is ONE counting-sort pass over an
// 18-bit key = direction cell (6 bits, 8x8 octahedral, major) | 12-bit Morton code of the origin in a 16^3 grid:
//   k_sort_hist    read o,d (32 B) -> key (4 B) + global histogram (262144 bins, L2-resident atomics)
//   k_sort_scan    one block per 32768 bins: exclusive scan of the histogram chunk + chunk total
//   k_sort_scatter read ray (72 B + key) -> slot = atomicAdd(bin) -> write ray (72 B)
// ~= 184 B/ray of HBM traffic, no multi-pass key shuffling.  Order inside a bin is arbitrary (and irrelevant).
#pragma once

#include "dev_buf.h"
#include "rt_kernels.cuh"

namespace rt {

// Allocated by rc_resize: keys / keys_sorted per ray of the frame, hist / chunk_totals once.
struct SortBufs {
    DevBuf<uint32_t> keys;         // key per input ray
    DevBuf<uint32_t> keys_sorted;  // key per output ray (diagnostics / stage API)
    DevBuf<uint32_t> hist;         // kMaxBounces x kSortBins: one histogram per ray list, zeroed once per sample
    DevBuf<uint32_t> chunk_totals; // kMaxBounces x kSortChunks (k_sort_scan -> k_sort_scatter)
    float root_min[3] = {0, 0, 0};
    float inv_cell[3] = {1, 1, 1};
};

inline void set_sort_bounds(SortBufs &s, const float bmin[3], const float bmax[3]) {
    for (int i = 0; i < 3; ++i) {
        s.root_min[i] = bmin[i];
        const float ext = bmax[i] - bmin[i];
        s.inv_cell[i] = (ext > 0.0f) ? float(1 << kSortCellBits) / ext : 0.0f;
    }
}

__global__ void __launch_bounds__(256) k_sort_hist(const uint32_t *counters, int bounce, RayBuf rays, SortGrid g,
                                                   uint32_t *keys, uint32_t *hist) {
    const uint32_t count = counters[CNT_RAYS + bounce];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const uint32_t key = ray_sort_key(rays.o_cw[i], rays.d_cs[i], g);
        keys[i] = key;
        atomicAdd(&hist[key], 1u);
    }
}

// Exclusive scan of kSortBins counters: one 1024-thread block per 32768-bin chunk, all chunks in parallel.  Each block
// scans its chunk locally (warp w owns bins [1024 w, 1024 (w+1)) of the chunk as 32 rows of 32: coalesced rows, shuffle
// scan inside a row) and publishes the chunk's total in chunk_totals[]; the scatter kernel adds the prefix of the totals
// of the chunks before the key's chunk, so no second pass and no inter-block wait is needed.
constexpr int kSortChunkBins = 32 * 1024;
constexpr int kSortChunks = kSortBins / kSortChunkBins;
static_assert(kSortBins % kSortChunkBins == 0 && kSortChunks <= 64, "whole chunks");

__global__ void __launch_bounds__(1024) k_sort_scan(uint32_t *hist, uint32_t *chunk_totals) {
    __shared__ uint32_t warp_sums[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t *row0 = hist + blockIdx.x * kSortChunkBins + warp * 1024 + lane;
    uint32_t excl[32];
    uint32_t running = 0;
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        const uint32_t v = row0[r * 32];
        uint32_t incl = v;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) {
                incl += u;
            }
        }
        excl[r] = running + incl - v;
        running += __shfl_sync(0xffffffffu, incl, 31);
    }
    if (lane == 0) {
        warp_sums[warp] = running;
    }
    __syncthreads();
    if (warp == 0) {
        const uint32_t t = warp_sums[lane];
        uint32_t w = t;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= off) {
                w += u;
            }
        }
        warp_sums[lane] = w - t;
        if (lane == 31) {
            chunk_totals[blockIdx.x] = w;
        }
    }
    __syncthreads();
    const uint32_t base = warp_sums[warp];
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        row0[r * 32] = base + excl[r];
    }
}

__global__ void __launch_bounds__(256) k_sort_scatter(const uint32_t *counters, int bounce, RayBuf src, RayBuf dst,
                                                      const uint32_t *keys, uint32_t *offsets,
                                                      const uint32_t *chunk_totals, uint32_t *keys_sorted) {
    __shared__ uint32_t chunk_base[kSortChunks];
    if (threadIdx.x == 0) {
        uint32_t acc = 0;
        for (int c = 0; c < kSortChunks; ++c) {
            chunk_base[c] = acc;
            acc += chunk_totals[c];
        }
    }
    __syncthreads();
    const uint32_t count = counters[CNT_RAYS + bounce];
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        const uint32_t key = keys[i];
        const uint32_t slot = chunk_base[key / kSortChunkBins] + atomicAdd(&offsets[key], 1u);
        dst.o_cw[slot] = src.o_cw[i];
        dst.d_cs[slot] = src.d_cs[i];
        dst.c_pdf[slot] = src.c_pdf[i];
        dst.ior[slot] = src.ior[i];
        dst.xy_depth[slot] = src.xy_depth[i];
        if (keys_sorted) {
            keys_sorted[slot] = key;
        }
    }
}

// Reorders list `bounce` from `src` into `dst` (caller swaps its notion of the current buffer).
// have_hist: keys and the histogram of this list were already produced by the kernel that wrote the list (k_shade, see
// KParams::sort_hist), so the 32 B/ray key pass is skipped; otherwise (stage API) they are built here.
inline void sort_rays(SortBufs &s, const KParams &p, const RayBuf &src, const RayBuf &dst, int bounce, int num_sms,
                      bool have_hist, bool want_sorted_keys, cudaStream_t stream) {
    uint32_t *hist = s.hist.get() + size_t(bounce) * kSortBins;
    if (!have_hist) {
        SortGrid g{s.root_min[0], s.root_min[1], s.root_min[2], s.inv_cell[0], s.inv_cell[1], s.inv_cell[2]};
        cudaMemsetAsync(hist, 0, kSortBins * sizeof(uint32_t), stream);
        k_sort_hist<<<num_sms * 8, 256, 0, stream>>>(p.counters, bounce, src, g, s.keys.get(), hist);
    }
    uint32_t *chunk_totals = s.chunk_totals.get() + size_t(bounce) * kSortChunks;
    k_sort_scan<<<kSortChunks, 1024, 0, stream>>>(hist, chunk_totals);
    k_sort_scatter<<<num_sms * 8, 256, 0, stream>>>(p.counters, bounce, src, dst, s.keys.get(), hist, chunk_totals,
                                                    want_sorted_keys ? s.keys_sorted.get() : nullptr);
}

} // namespace rt
