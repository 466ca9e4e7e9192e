// rt_ppm.cu — output_to_stream (main.cu:321-333) on the device: the frame is quantised and formatted as P3 text in HBM,
// only the text crosses PCIe.
//
// The reference streams `int(255.99 * channel)` token by token from managed memory through an ostream — ~12 bytes of text
// per pixel, 0.4 s of host time for a 3840x2160 frame even with a hand-rolled itoa (rt_format_ppm, the host writer kept
// for small frames and as the checker).  Variable-length records make it a scan problem:
//   k_ppm_len    one thread per pixel in OUTPUT order (rows top to bottom, j = ny-1 .. 0): text length of the pixel's line,
//                block-reduced to one length per 256 pixels
//   k_ppm_scan   exclusive scan of the block lengths (one block; 32 k values at 4K)
//   k_ppm_write  recomputes the three integers, block-scans the line lengths, formats the block's lines into shared memory
//                at the same 16-byte phase as their destination and streams them out with 16-byte stores
// HBM-bound byte work: reads 2 x 12 B/pixel, writes ~11.5 B/pixel of text (bench: profiles/).  The bytes are identical to
// the host writer's for every finite input; like the x86 cast the reference relies on, out-of-range and NaN values print
// INT_MIN.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "rt_render.h"

namespace rt {

constexpr int kPpmThreads = 256;
constexpr int kPpmMaxLine = 36;      // "-2147483648 -2147483648 -2147483648\n"

struct PpmHead {
    char text[64];
    int len;
};

// int(255.99 * double(v)) with the x86 behaviour for values a 32-bit int cannot hold (cvttsd2si -> 0x80000000)
__device__ __forceinline__ int ppm_quantise(const float v) {
    const double x = 255.99 * (double)v;
    if (!(fabs(x) < 2147483648.0)) return (int)0x80000000u;
    return __double2int_rz(x);
}
__device__ __forceinline__ int ppm_digits(const int v) {      // characters `ostream << v` prints
    const unsigned u = v < 0 ? 0u - (unsigned)v : (unsigned)v;
    int n = 1 + (v < 0);
    n += (u >= 10u) + (u >= 100u) + (u >= 1000u) + (u >= 10000u) + (u >= 100000u) + (u >= 1000000u) + (u >= 10000000u) +
         (u >= 100000000u) + (u >= 1000000000u);
    return n;
}
__device__ __forceinline__ char *ppm_put(char *p, const int v, const int n) {
    unsigned u = v < 0 ? 0u - (unsigned)v : (unsigned)v;
    char *q = p + n;
    do { *--q = (char)('0' + u % 10u); u /= 10u; } while (u);
    if (v < 0) *--q = '-';
    return p + n;
}
// pixel t of the text (row-major from the TOP row) -> the frame's pixel (rows bottom to top, main.cu:323)
__device__ __forceinline__ size_t ppm_source(const size_t t, const int nx, const int ny) {
    const size_t row = t / (size_t)nx, i = t - row * (size_t)nx;
    return ((size_t)(ny - 1) - row) * (size_t)nx + i;
}

__device__ __forceinline__ uint32_t block_sum(uint32_t v, uint32_t *warp_sums) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) warp_sums[threadIdx.x >> 5] = v;
    __syncthreads();
    uint32_t s = 0;
    for (int w = 0; w < kPpmThreads / 32; w++) s += warp_sums[w];
    return s;
}

__global__ void __launch_bounds__(kPpmThreads) k_ppm_len(const float *__restrict__ fb, int nx, int ny, size_t npix, uint32_t *__restrict__ block_len) {
    __shared__ uint32_t warp_sums[kPpmThreads / 32];
    const size_t t = (size_t)blockIdx.x * kPpmThreads + threadIdx.x;
    uint32_t len = 0;
    if (t < npix) {
        const float *px = fb + ppm_source(t, nx, ny) * 3;
        len = 3u + ppm_digits(ppm_quantise(px[0])) + ppm_digits(ppm_quantise(px[1])) + ppm_digits(ppm_quantise(px[2]));
    }
    const uint32_t s = block_sum(len, warp_sums);
    if (threadIdx.x == 0) block_len[blockIdx.x] = s;
}

// exclusive scan of n block lengths into 64-bit offsets starting at `first`; off[n] = total
__global__ void __launch_bounds__(1024) k_ppm_scan(const uint32_t *__restrict__ len, size_t n, unsigned long long first, unsigned long long *__restrict__ off) {
    __shared__ unsigned long long warp_tot[32];
    const size_t per = (n + 1023) / 1024, b = threadIdx.x * per, e = b + per < n ? b + per : n;
    unsigned long long s = 0;
    for (size_t k = b; k < e; k++) s += len[k];
    // exclusive block scan of the per-thread sums: shuffles inside a warp, then the 32 warp totals
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    unsigned long long incl = s;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += v;
    }
    if (lane == 31u) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        unsigned long long t = warp_tot[lane], ti = t;
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, ti, o);
            if (lane >= (unsigned)o) ti += v;
        }
        warp_tot[lane] = ti - t;                    // exclusive
        if (lane == 31u) off[n] = first + ti;       // total text length
    }
    __syncthreads();
    unsigned long long acc = first + warp_tot[warp] + (incl - s);
    for (size_t k = b; k < e; k++) { off[k] = acc; acc += len[k]; }
}

__global__ void __launch_bounds__(kPpmThreads) k_ppm_write(const float *__restrict__ fb, int nx, int ny, size_t npix,
                                                           const unsigned long long *__restrict__ block_off, const __grid_constant__ PpmHead head,
                                                           char *__restrict__ text) {
    __shared__ __align__(16) char buf[kPpmThreads * kPpmMaxLine + 16];
    __shared__ uint32_t warp_sums[kPpmThreads / 32];
    const size_t t = (size_t)blockIdx.x * kPpmThreads + threadIdx.x;
    int q[3] = {0, 0, 0}, nd[3] = {0, 0, 0};
    uint32_t len = 0;
    if (t < npix) {
        const float *px = fb + ppm_source(t, nx, ny) * 3;
#pragma unroll
        for (int k = 0; k < 3; k++) { q[k] = ppm_quantise(px[k]); nd[k] = ppm_digits(q[k]); }
        len = 3u + nd[0] + nd[1] + nd[2];
    }
    // exclusive scan of the line lengths over the block
    const unsigned lane = threadIdx.x & 31u;
    uint32_t incl = len;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= (unsigned)o) incl += v;
    }
    if (lane == 31u) warp_sums[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (int w = 0; w < kPpmThreads / 32; w++) {
        const uint32_t s = warp_sums[w];
        if (w < (int)(threadIdx.x >> 5)) before += s;
        total += s;
    }
    const unsigned long long dst0 = block_off[blockIdx.x];
    const uint32_t phase = (uint32_t)(dst0 & 15ull);          // shared-memory position p <-> text[dst0 - phase + p]
    if (len) {
        char *p = buf + phase + before + (incl - len);
        p = ppm_put(p, q[0], nd[0]); *p++ = ' ';
        p = ppm_put(p, q[1], nd[1]); *p++ = ' ';
        p = ppm_put(p, q[2], nd[2]); *p++ = '\n';
    }
    __syncthreads();
    char *dst = text + (dst0 - phase);
    const uint32_t b = phase, e = phase + total;
    const uint32_t vb = (b + 15u) & ~15u, ve = e & ~15u;       // the 16-byte-aligned body
    if (vb < ve) {
        for (uint32_t k = threadIdx.x; k < vb - b; k += kPpmThreads) dst[b + k] = buf[b + k];
        for (uint32_t k = vb + 16u * threadIdx.x; k < ve; k += 16u * kPpmThreads)
            *reinterpret_cast<uint4 *>(dst + k) = *reinterpret_cast<const uint4 *>(buf + k);
        for (uint32_t k = ve + threadIdx.x; k < e; k += kPpmThreads) dst[k] = buf[k];
    } else {
        for (uint32_t k = b + threadIdx.x; k < e; k += kPpmThreads) dst[k] = buf[k];
    }
    if (blockIdx.x == 0 && threadIdx.x < (unsigned)head.len) text[threadIdx.x] = head.text[threadIdx.x];
}

// formats fb (device, nx*ny*3 floats) into ws.text; returns the text length through *len_out (synchronises the stream once)
cudaError_t ppm_format_device(PpmWorkspace &ws, const float *fb, int nx, int ny, cudaStream_t st, size_t *len_out) {
    const size_t npix = (size_t)nx * ny;
    const size_t blocks = (npix + kPpmThreads - 1) / kPpmThreads;
    cudaError_t e;
    if ((e = ws.block_len.reserve(blocks + 1)) != cudaSuccess || (e = ws.block_off.reserve(blocks + 1)) != cudaSuccess) return e;
    PpmHead head;
    head.len = snprintf(head.text, sizeof head.text, "P3\n%d %d\n255\n", nx, ny);
    if (blocks) k_ppm_len<<<(unsigned)blocks, kPpmThreads, 0, st>>>(fb, nx, ny, npix, ws.block_len.ptr);
    k_ppm_scan<<<1, 1024, 0, st>>>(ws.block_len.ptr, blocks, (unsigned long long)head.len, ws.block_off.ptr);
    unsigned long long total = 0;
    if ((e = cudaMemcpyAsync(&total, ws.block_off.ptr + blocks, sizeof total, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    if ((e = ws.text.reserve(total + 16)) != cudaSuccess) return e;
    if (blocks) {
        k_ppm_write<<<(unsigned)blocks, kPpmThreads, 0, st>>>(fb, nx, ny, npix, ws.block_off.ptr, head, ws.text.ptr);
    } else {
        if ((e = cudaMemcpyAsync(ws.text.ptr, head.text, (size_t)head.len, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    }
    ws.text_len = (size_t)total;
    if (len_out) *len_out = (size_t)total;
    return cudaGetLastError();
}

}  // namespace rt
