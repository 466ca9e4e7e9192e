// rt_adaptive.h — adaptive sampling (rt_render_adaptive): the per-pixel noise estimate, and the launch interface of the selection
// pass (rt_adaptive.cu).
//
// The render kernels keep linear sums only, so there is no per-sample variance.  The estimate compares two independent segments
// of a pixel's own sample chain: A = samples [0, a), read from a snapshot of the sum, and B = samples [a, c), the current sum minus
// that snapshot.  d is the largest per-channel difference of the two segment means in display space (the frame is sqrt(mean)); w
// scales it to the standard error of the combined c-sample mean (Var(A - B) = sigma^2 c / (a b)).  Every operation is an
// explicitly rounded IEEE float operation (rt_math.cuh), so a host build with -ffp-contract=off gives the same bits.  A NaN
// result (a non-finite sum) counts as not converged.
#pragma once
#include <stdint.h>

#include "rt_math.cuh"

namespace rt {

// e_p of a pixel: s = snapshot sum after a samples, x = current sum after c > a samples
RT_HD float adaptive_error(const float s[3], uint32_t a, const float x[3], uint32_t c) {
    const float fa = (float)a, fb = (float)(c - a);
    float d = 0.0f;
    for (int k = 0; k < 3; k++) {
        const float A = div_(s[k], fa), B = div_(sub_(x[k], s[k]), fb);
        const float dk = fabsf(sub_(sqrt_(A), sqrt_(B)));
        d = (k == 0 || dk > d || dk != dk) ? dk : d;          // max of the three, NaN propagating (as numpy.maximum)
    }
    const float w = div_(mul_(sqrt_(fa), sqrt_(fb)), (float)c);
    return mul_(d, w);
}

#if defined(__CUDACC__)
// Per-tile scratch of the selection pass, owned by the context: tiles = ceil(nx/8) * ceil(ny/4) tiles of the frame queue
struct AdaptiveTiles {
    uint32_t *listed;        // pixels tile t lists this round (its in-frame pixels if refined, else 0)
    uint32_t *offset;        // inclusive prefix sum of `listed`
    uint32_t *done;          // 1: the tile is never evaluated again
    void *scan_temp;         // cub::DeviceScan temporary storage
    size_t scan_temp_bytes;
};
// bytes of cub temporary storage the scan over `tiles` tiles needs
cudaError_t adaptive_scan_temp_bytes(uint32_t tiles, size_t *bytes);
// counts[i] = value for npix pixels
cudaError_t launch_fill_counts(uint32_t *counts, size_t npix, uint32_t value, cudaStream_t st);
// One selection round over the tiles not done.  Every pixel of such a tile has snapshot count a and count c; with refine_ok (c <
// max_spp) a tile whose largest e_p is not <= threshold is refined: its snapshot becomes its sum and its in-frame pixels are
// appended to `list` (tiles row-major, pixels row by row inside a tile); any other evaluated tile is done.  err (optional) receives
// e_p of every evaluated pixel.  *listed_host: the length of the list (read back: the call waits for the stream).
cudaError_t launch_adaptive_select(const float *accum, float *snap, float *err, int nx, int ny, uint32_t a, uint32_t c, bool refine_ok,
                                   float threshold, const AdaptiveTiles &t, uint32_t *list, uint32_t *listed_host, cudaStream_t st);
#endif

}  // namespace rt
