// rt_adaptive.cu — the selection pass of rt_render_adaptive: which 8x4 tiles of the frame queue get more samples in a round, and
// their pixel list in a deterministic order for the list-progressive render kernels.
//
// Three launches per round that can refine:
//   k_adaptive_select  one warp per tile, one lane per pixel: a done tile reads its flag and leaves; any other tile evaluates e_p
//                      (rt_adaptive.h) of its in-frame pixels, reduces the largest by bit pattern (e_p >= 0; NaN counts as +inf)
//                      and decides.  A refined tile takes its sums as its new snapshot and records how many pixels it lists;
//                      any other tile is done for good (its inputs can no longer change);
//   cub::DeviceScan    inclusive sum of the per-tile pixel counts: each refined tile's slot in the list;
//   k_adaptive_emit    one warp per refined tile writes its in-frame pixels, row by row, at its slot.
// The list is window_pixels(nx, ny, 0, nx, 0, ny) restricted to the refined tiles: whole, coherent tiles, in an order no atomic
// decides.  Its length crosses to the host once per round.
#include <cuda_runtime.h>
#include <stdint.h>

#include <cub/device/device_scan.cuh>

#include "rt_adaptive.h"

namespace rt {

constexpr int kSelectThreads = 256;      // 8 tiles per block

__device__ __forceinline__ bool tile_pixel(uint32_t tile, int lane, int nx, int ny, int tiles_x, uint32_t &pix) {
    const uint32_t ty = tile / (uint32_t)tiles_x, tx = tile - ty * (uint32_t)tiles_x;
    const int i = (int)(tx * 8u) + (lane & 7), j = (int)(ty * 4u) + (lane >> 3);
    pix = (uint32_t)j * (uint32_t)nx + (uint32_t)i;
    return i < nx && j < ny;
}

__global__ void __launch_bounds__(kSelectThreads) k_adaptive_select(const float *__restrict__ accum, float *__restrict__ snap,
                                                                    float *__restrict__ err, int nx, int ny, int tiles_x, uint32_t tiles,
                                                                    uint32_t a, uint32_t c, int refine_ok, float threshold,
                                                                    uint32_t *__restrict__ listed, uint32_t *__restrict__ done) {
    const uint32_t tile = (blockIdx.x * kSelectThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (tile >= tiles) return;                       // (whole warps)
    if (done[tile]) {
        if (lane == 0) listed[tile] = 0;
        return;
    }
    uint32_t pix;
    const bool in = tile_pixel(tile, lane, nx, ny, tiles_x, pix);
    float x[3] = {0.f, 0.f, 0.f};
    uint32_t bits = 0;                               // out-of-frame lanes: +0, below every e_p
    if (in) {
        float s[3];
        for (int k = 0; k < 3; k++) { x[k] = accum[(size_t)pix * 3 + k]; s[k] = snap[(size_t)pix * 3 + k]; }
        const float e = adaptive_error(s, a, x, c);
        if (err) err[pix] = e;
        bits = e != e ? 0x7f800000u : __float_as_uint(e);
    }
    const float tile_err = __uint_as_float(__reduce_max_sync(0xffffffffu, bits));
    const bool refine = refine_ok && !(tile_err <= threshold);
    const uint32_t n_in = (uint32_t)__popc(__ballot_sync(0xffffffffu, in));
    if (refine && in)
        for (int k = 0; k < 3; k++) snap[(size_t)pix * 3 + k] = x[k];
    if (lane == 0) {
        listed[tile] = refine ? n_in : 0u;
        if (!refine) done[tile] = 1u;
    }
}

__global__ void __launch_bounds__(kSelectThreads) k_adaptive_emit(int nx, int ny, int tiles_x, uint32_t tiles, const uint32_t *__restrict__ listed,
                                                                  const uint32_t *__restrict__ offset, uint32_t *__restrict__ list) {
    const uint32_t tile = (blockIdx.x * kSelectThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (tile >= tiles) return;
    const uint32_t n = listed[tile];
    if (n == 0) return;
    uint32_t pix;
    const bool in = tile_pixel(tile, lane, nx, ny, tiles_x, pix);
    const uint32_t below = __ballot_sync(0xffffffffu, in) & ((1u << lane) - 1u);     // in-frame lanes before this one (row by row)
    if (in) list[offset[tile] - n + (uint32_t)__popc(below)] = pix;
}

__global__ void k_fill_counts(uint32_t *__restrict__ counts, size_t npix, uint32_t value) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npix) counts[i] = value;
}

cudaError_t adaptive_scan_temp_bytes(uint32_t tiles, size_t *bytes) {
    *bytes = 0;
    return cub::DeviceScan::InclusiveSum(nullptr, *bytes, static_cast<const uint32_t *>(nullptr), static_cast<uint32_t *>(nullptr), (int)tiles);
}

cudaError_t launch_fill_counts(uint32_t *counts, size_t npix, uint32_t value, cudaStream_t st) {
    k_fill_counts<<<(unsigned)((npix + 255) / 256), 256, 0, st>>>(counts, npix, value);
    return cudaGetLastError();
}

cudaError_t launch_adaptive_select(const float *accum, float *snap, float *err, int nx, int ny, uint32_t a, uint32_t c, bool refine_ok,
                                   float threshold, const AdaptiveTiles &t, uint32_t *list, uint32_t *listed_host, cudaStream_t st) {
    const int tiles_x = (nx + 7) / 8;
    const uint32_t tiles = (uint32_t)tiles_x * (uint32_t)((ny + 3) / 4);
    const unsigned blocks = (unsigned)((tiles + kSelectThreads / 32 - 1) / (kSelectThreads / 32));
    k_adaptive_select<<<blocks, kSelectThreads, 0, st>>>(accum, snap, err, nx, ny, tiles_x, tiles, a, c, refine_ok ? 1 : 0, threshold,
                                                         t.listed, t.done);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    *listed_host = 0;
    if (!refine_ok) return cudaSuccess;              // nothing can be listed: every evaluated tile is done
    size_t temp = t.scan_temp_bytes;
    e = cub::DeviceScan::InclusiveSum(t.scan_temp, temp, t.listed, t.offset, (int)tiles, st);
    if (e != cudaSuccess) return e;
    k_adaptive_emit<<<blocks, kSelectThreads, 0, st>>>(nx, ny, tiles_x, tiles, t.listed, t.offset, list);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(listed_host, t.offset + (tiles - 1), 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    return cudaStreamSynchronize(st);
}

}  // namespace rt
