// rt_render.cu — the render hot path: render_init + render + color (main.cu:43-117) as ONE persistent kernel.
//
// Reference shape: thread = pixel, 8x8 blocks, each thread runs its ns samples x <=50 bounces serially, so a warp
// lives as long as its slowest pixel and every bounce pays two virtual calls and an AoS pointer chase.
// This kernel:
//   * persistent threads: the grid is sized to what is resident on the SMs; every lane owns one pixel chain at a time and
//     claims the next pixel from a queue when it is done (the lane loop of rt_chain.cuh, shared with k_render_coop);
//   * pixels are queued in 8x4 tiles so that the 32 lanes of a warp start on neighbouring pixels (coherent rays);
//   * XORWOW state lives in registers and is seeded in place (render_init fused; no 48-byte state array);
//   * spheres are SoA float4, materials are tag-dispatched (no device heap, no vtables);
//   * octree mode never walks the tree: one uniform grid + the reference's cell-visibility rule (rt_trace.cuh);
//   * flat-list mode stages the whole float4 sphere array once per block in shared memory with a TMA bulk copy
//     (cp.async.bulk + mbarrier) and sweeps it with warp-uniform (broadcast) shared-memory reads.
#include <cuda_runtime.h>
#include <stdint.h>

#include "rt_render.h"
#include "rt_build.cuh"
#include "rt_half.cuh"
#include "rt_trace.cuh"
#include "rt_xorwow_skip.h"

namespace rt {

// The camera is per-CONTEXT state: it travels in the launch parameters (RenderLaunch::cam, constant bank), not in a
// per-library __constant__ symbol that two contexts on one GPU would overwrite for each other.

// ---- TMA 1-D bulk copy global -> shared, completion on an mbarrier -------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    // bounded: a copy of a few KB completes in microseconds; never spin forever on a broken descriptor
    for (int spin = 0; spin < (1 << 22) && !done; spin++) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
    if (!done) __trap();
}

// Stage `bytes` (multiple of 16, 16-byte aligned on both sides) in chunks the bulk-copy engine accepts.
__device__ __forceinline__ void stage_bulk(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    const uint32_t kChunk = 32768;
    for (uint32_t off = 0; off < bytes; off += kChunk) {
        const uint32_t n = bytes - off < kChunk ? bytes - off : kChunk;
        bulk_g2s(static_cast<char *>(dst) + off, static_cast<const char *>(src) + off, n, bar);
    }
}

// render_init (main.cu:84-94): the pixel's XORWOW stream.  HEAD seeding curand_init(1984 + pixel_index, 0, 0) is a dozen
// integer operations and happens right here; the upstream form curand_init(1984, pixel_index, 0) needs the skip-ahead
// and is precomputed per pixel by k_seed_upstream.
__device__ __forceinline__ void pixel_stream(const RenderLaunch &p, const int pix, xorwow &rng) {
    if (p.seed_states) {
        const uint2 *s = reinterpret_cast<const uint2 *>(p.seed_states + (size_t)pix * 6);
        const uint2 a = __ldg(s), b = __ldg(s + 1), c = __ldg(s + 2);
        rng.d = a.x; rng.v0 = a.y; rng.v1 = b.x; rng.v2 = b.y; rng.v3 = c.x; rng.v4 = c.y;
    } else {
        xorwow_seed(rng, (unsigned long long)(long long)(1984 + pix) + p.seed_offset);   // main.cu:93
    }
}

__global__ void k_seed_upstream(uint32_t *__restrict__ states, size_t npix, unsigned long long seed, unsigned long long base,
                                const uint32_t *__restrict__ tables) {
    const size_t pix = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= npix) return;
    xorwow s;
    xorwow_seed_subsequence(s, seed, base + pix, tables);
    xorwow_store(states + pix * 6, s);
}

cudaError_t launch_seed_upstream(uint32_t *states, size_t npix, unsigned long long seed, unsigned long long subsequence_base,
                                 const uint32_t *tables, cudaStream_t st) {
    k_seed_upstream<<<(unsigned)((npix + 127) / 128), 128, 0, st>>>(states, npix, seed, subsequence_base, tables);
    return cudaGetLastError();
}

// upstream seeding of a pixel list: entry k gets the stream of pixel pixels[k] (count x 24 bytes, not one state per frame pixel)
__global__ void k_seed_upstream_list(uint32_t *__restrict__ states, const uint32_t *__restrict__ pixels, int count, size_t npix,
                                     unsigned long long seed, const uint32_t *__restrict__ tables) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const uint32_t pix = pixels[k];
    if (pix >= npix) return;                  // out of the frame: never traced, its state is never read
    xorwow s;
    xorwow_seed_subsequence(s, seed, pix, tables);
    xorwow_store(states + (size_t)k * 6, s);
}

cudaError_t launch_seed_upstream_list(uint32_t *states, const uint32_t *pixels, int count, size_t npix, unsigned long long seed,
                                      const uint32_t *tables, cudaStream_t st) {
    k_seed_upstream_list<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(states, pixels, count, npix, seed, tables);
    return cudaGetLastError();
}

// The preparation pass of rt_render_pixels_progressive, one thread per list entry:
//   * dedupe: the entry that sets its pixel's bit in `mask` (npix bits, zero on entry) keeps the pixel in `filtered`; an entry
//     outside the frame and every later duplicate become 0xFFFFFFFF there, so the list keeps its order (and its warps their
//     neighbouring pixels).  Which duplicate wins does not matter: each would do the same work on the same pixel.  Without it two
//     lanes could hold one pixel, and the one that claims it late would resume the sum and stream the other has advanced;
//   * counts[pix] += ns (= ns when first) for the pixels kept, if counts is given;
//   * first: the kept pixels' streams are started in `states` (HEAD: seed 1984 + pix; UPSTREAM: curand_init(1984, pix, 0) with
//     the skip tables), so the render always resumes from `states`.
__global__ void k_pixels_progressive_prep(const uint32_t *__restrict__ pixels, int count, uint32_t npix, uint32_t *__restrict__ mask,
                                          uint32_t *__restrict__ filtered, uint32_t *__restrict__ counts, uint32_t ns, int first,
                                          uint32_t *__restrict__ states, const uint32_t *__restrict__ tables) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const uint32_t e = pixels[k];
    bool keep = e < npix;
    if (keep) {
        const uint32_t bit = 1u << (e & 31u);
        keep = !(atomicOr(mask + (e >> 5), bit) & bit);
    }
    filtered[k] = keep ? e : 0xFFFFFFFFu;
    if (!keep) return;
    if (counts) counts[e] = first ? ns : counts[e] + ns;
    if (first) {
        xorwow s;
        if (tables) xorwow_seed_subsequence(s, 1984ull, e, tables);
        else xorwow_seed(s, 1984ull + e);      // main.cu:93, as pixel_stream
        xorwow_store(states + (size_t)e * 6, s);
    }
}

cudaError_t launch_pixels_progressive_prep(const uint32_t *pixels, int count, uint32_t npix, uint32_t *mask, uint32_t *filtered, uint32_t *counts,
                                           uint32_t ns, bool first, uint32_t *states, const uint32_t *upstream_tables, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(mask, 0, (size_t)(npix + 31) / 32 * 4, st);
    if (e != cudaSuccess) return e;
    k_pixels_progressive_prep<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(pixels, count, npix, mask, filtered, counts, ns, first ? 1 : 0,
                                                                                states, upstream_tables);
    return cudaGetLastError();
}

// item -> pixel.  Items enumerate 8x4 tiles row-major, 32 pixels per tile; `tile_stride/tile_first` select the
// interleaved tiles a shard owns (RT_SHARD_TILES).
__device__ __forceinline__ bool item_to_pixel(const RenderLaunch &p, uint32_t item, int &i, int &j) {
    const uint32_t local_tile = item >> 5, in = item & 31u;
    const uint32_t tile = local_tile * (uint32_t)p.tile_stride + (uint32_t)p.tile_first;
    const uint32_t ty = tile / (uint32_t)p.tiles_x, tx = tile - ty * (uint32_t)p.tiles_x;
    i = (int)(tx * 8u + (in & 7u));
    j = (int)(ty * 4u + (in >> 3));
    return i < p.nx && j < p.ny;
}

// item -> pixel of a pixel-list launch (kModeList / kModeListProgressive instances): item k is list entry k, so a warp starts on
// 32 consecutive entries.  kModeList: the claiming lane keeps k as its slot (result at out[3k], upstream start state at
// seed_states[6k]); camera u, v and the HEAD seed use the pixel's frame coordinates.  An entry outside the frame is not traced;
// with zero_outside (kModeList, whose `out` is in list order) it gets (0, 0, 0) — kModeListProgressive's `out` is the caller's
// frame, where such an entry owns nothing.
__device__ __forceinline__ bool list_to_pixel(const RenderLaunch &p, uint32_t item, int &i, int &j, const bool zero_outside) {
    const uint32_t e = __ldg(p.pixels + item);
    if ((unsigned long long)e >= (unsigned long long)p.nx * (unsigned long long)p.ny) {
        if (zero_outside) {
            float *out = p.out + (size_t)item * 3;
            out[0] = 0.0f; out[1] = 0.0f; out[2] = 0.0f;
        }
        return false;
    }
    j = (int)(e / (uint32_t)p.nx);
    i = (int)(e - (uint32_t)j * (uint32_t)p.nx);
    return true;
}

// Queue pop for the lanes in `m` (ballot of the lanes that need a pixel), compacted per warp and served from the WARP'S
// OWN stock of whole tiles: [stock_next, stock_end) is the unclaimed rest of the last tile this warp took from the
// frame-wide queue (one atomicAdd of `batch` items when it runs out).  A lane that finishes its pixel continues inside
// its warp's tile, so the rays of a warp stay neighbours in the image however long the sample chains are (with one
// pixel-granular queue they drift apart: lanes finish one at a time, wherever the frame-wide head happens to be).
// batch = 1 restores that queue — for frames with only a few pixels per lane, where the tail of the frame is what counts.
// Every lane of the warp calls; the result is meaningful for the lanes in m.
__device__ __forceinline__ uint32_t claim_items(const RenderLaunch &p, const unsigned m, const unsigned lane, uint32_t &stock_next,
                                                uint32_t &stock_end, const uint32_t batch) {
    const uint32_t k = (uint32_t)__popc(m), rank = (uint32_t)__popc(m & ((1u << lane) - 1u)), avail = stock_end - stock_next;
    uint32_t item = stock_next + rank;
    if (k <= avail) {
        stock_next += k;
    } else {
        const uint32_t need = k - avail, claim = (need + batch - 1u) / batch * batch;
        uint32_t base = 0;
        const int leader = __ffs(m) - 1;
        if ((int)lane == leader) base = atomicAdd(p.work_counter, claim);
        base = __shfl_sync(0xffffffffu, base, leader);
        if (rank >= avail) item = base + (rank - avail);
        stock_next = base + need;
        stock_end = base + claim;
    }
    return item;
}
__device__ __forceinline__ uint32_t claim_batch(const RenderLaunch &p) {   // pixels per lane decide: whole tiles, or single pixels
    if (p.variant == 31) return 1u;          // A/B: the frame-wide pixel queue
    return p.total_items / (gridDim.x * blockDim.x) >= 4u ? 32u : 1u;
}

#include "rt_chain.cuh"

// The body of k_render and k_render_pixels_progressive; MODE: rt_render.h LaunchMode (what the queue's items are, run_chains).
template <bool OCTREE, bool GEOM_SMEM, int MODE>
__device__ __forceinline__ void render_lanes(const RenderLaunch &p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ __align__(8) uint64_t bar;

    // ---- flat-list mode: stage the whole float4 sphere array in shared memory with a TMA bulk copy ----
    const SceneView sc = p.scene;
    const float4 *geom_s = nullptr;
    if (!OCTREE && GEOM_SMEM) {
        const uint32_t total = (uint32_t)sc.n * sizeof(float4);
        if (threadIdx.x == 0) {
            mbar_init(&bar, 1);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(&bar, total);
            stage_bulk(smem_raw, p.scene.geom, total, &bar);
        }
        geom_s = reinterpret_cast<const float4 *>(smem_raw);
        mbar_wait(&bar, 0);
    }

    TraceCounters tc;
    tc.sphere_tests = tc.node_tests = tc.voxel_steps = 0;
    run_chains<MODE>(p, ChainF32(p), claim_batch(p), [&](Chain &c, const bool has) {
        Hit h;
        if (has) {   // per lane: only the lanes that hold a pixel trace
            if (OCTREE) h = trace_tree(sc, p.tree, &p.tree.planes[0][0], c.o, c.d, tc);
            else if (GEOM_SMEM) h = trace_list(geom_s, sc.tag, sc.n, c.o, c.d, tc);
            else h = trace_list(sc.geom, sc.tag, sc.n, c.o, c.d, tc);
        }
        return h;
    });
#ifdef RT_COUNTERS
    const unsigned lane = threadIdx.x & 31u;
    unsigned long long c64[3] = {tc.sphere_tests, tc.node_tests, tc.voxel_steps};
    for (int k = 0; k < 3; k++) {
        for (int off = 16; off > 0; off >>= 1) c64[k] += __shfl_xor_sync(0xffffffffu, c64[k], off);
        if (lane == 0) atomicAdd(p.counters + 2 + k, c64[k]);
    }
#endif
}

// LIST: pixel-list instances (rt_render_pixels, list_to_pixel); a chain's `pix` is then the lane's list slot.
template <bool OCTREE, bool GEOM_SMEM, bool LIST = false>
__global__ void __launch_bounds__(kRenderThreads, 6) k_render(const __grid_constant__ RenderLaunch p) {
    render_lanes<OCTREE, GEOM_SMEM, LIST ? kModeList : kModeFrame>(p);
}
// progressive pixel lists (rt_render_pixels_progressive): a chain's `pix` is the frame pixel, its sum and stream the frame's
template <bool OCTREE, bool GEOM_SMEM>
__global__ void __launch_bounds__(kRenderThreads, 6) k_render_pixels_progressive(const __grid_constant__ RenderLaunch p) {
    render_lanes<OCTREE, GEOM_SMEM, kModeListProgressive>(p);
}

// Persistent grid of a queue-fed render kernel: exactly the blocks that are resident, never more than there is work; the queue
// head starts past the grid (the first tile of every warp needs no atomic).  `args` are the kernel's arguments.
template <typename... Params, typename... Args>
static cudaError_t launch_persistent(void (*kern)(Params...), size_t smem, const RenderLaunch &p, int sm_count, cudaStream_t st,
                                     int *blocks_out, Args... args) {
    cudaError_t e;
    if (smem && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRenderThreads, smem);
    if (e != cudaSuccess) return e;
    if (per_sm < 1) return cudaErrorLaunchOutOfResources;
    long long blocks = (long long)per_sm * sm_count;
    const long long need = ((long long)p.total_items + kRenderThreads - 1) / kRenderThreads;
    if (blocks > need) blocks = need < 1 ? 1 : need;
    const uint32_t head = (uint32_t)(blocks * kRenderThreads);
    e = cudaMemcpyAsync(p.work_counter, &head, 4, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    kern<<<(unsigned)blocks, kRenderThreads, smem, st>>>(args...);
    if (blocks_out) *blocks_out = (int)blocks;
    return cudaGetLastError();
}

#include "rt_coop.cuh"
#include "rt_render_half.cuh"

cudaError_t launch_scene_to_half(const float4 *geom, const float4 *matl, int n, uint2 *geom_h, uint2 *matl_h, cudaStream_t st) {
    h16::k_scene_to_half<<<(n + 255) / 256, 256, 0, st>>>(geom, matl, n, geom_h, matl_h);
    return cudaGetLastError();
}
cudaError_t launch_camera_setup_half(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov, int nx, int ny,
                                     float aspect_override, float aperture, float focus_dist, __half *cam_h, cudaStream_t st) {
    h16::k_camera_setup_h<<<1, 1, 0, st>>>(lookfrom[0], lookfrom[1], lookfrom[2], lookat[0], lookat[1], lookat[2], vup[0], vup[1], vup[2],
                                           vfov, nx, ny, aspect_override, aperture, focus_dist, cam_h);
    return cudaGetLastError();
}
// the half kernels' views of the context's USE_FP16 pair lists and node tables
static void half_views(const HalfPairs &hp, h16::PairView &pv, h16::NodeTab &nt) {
    pv.geom = hp.geom.ptr; pv.idx = hp.idx.ptr; pv.start = hp.start.ptr;
    nt.ent = hp.nodes.ptr; nt.count = hp.node_count.ptr;
}
cudaError_t launch_render_half(const RenderLaunch &p, bool octree, const uint2 *geom_h, const uint2 *matl_h, const __half *cam_h,
                               const HalfPairs &hp, int sm_count, cudaStream_t st, int *blocks_out, int mode) {
    h16::PairView pv;
    h16::NodeTab nt;
    half_views(hp, pv, nt);
    const bool prog = p.accumulate || p.state_out;
    auto kern = mode == kModeListProgressive ? (octree ? h16::k_render_h<true, true, true> : h16::k_render_h<false, true, true>)
              : mode == kModeList ? (octree ? h16::k_render_h<true, false, true> : h16::k_render_h<false, false, true>)
              : octree ? (prog ? h16::k_render_h<true, true> : h16::k_render_h<true, false>)
                       : (prog ? h16::k_render_h<false, true> : h16::k_render_h<false, false>);
    return launch_persistent(kern, 0, p, sm_count, st, blocks_out, p, geom_h, matl_h, cam_h, pv, nt);
}

cudaError_t launch_finalize_half(const float *accum, float *fb, size_t count, int ns, cudaStream_t st) {
    h16::k_finalize_h<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(accum, fb, count, ns);
    return cudaGetLastError();
}

// fb = sqrt(sum * (1/counts[pix])) with ChainF32's reciprocal (1/S rounded once): what k_render writes for a pixel rendered with
// ns = counts[pix]; count 0 gives (0, 0, 0)
__global__ void k_finalize_counts(const float *__restrict__ accum, const uint32_t *__restrict__ counts, float *__restrict__ fb, size_t npix) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const uint32_t c = counts[i];
    const float a0 = accum[3 * i], a1 = accum[3 * i + 1], a2 = accum[3 * i + 2];
    if (c == 0) {
        fb[3 * i] = 0.0f; fb[3 * i + 1] = 0.0f; fb[3 * i + 2] = 0.0f;
        return;
    }
    const float inv_ns = __fdiv_rn(1.0f, (float)c);
    fb[3 * i] = sqrt_(mul_(a0, inv_ns));
    fb[3 * i + 1] = sqrt_(mul_(a1, inv_ns));
    fb[3 * i + 2] = sqrt_(mul_(a2, inv_ns));
}

cudaError_t launch_finalize_counts(const float *accum, const uint32_t *counts, float *fb, size_t npix, bool fp16, cudaStream_t st) {
    const unsigned blocks = (unsigned)((npix + 255) / 256);
    if (fp16) h16::k_finalize_counts_h<<<blocks, 256, 0, st>>>(accum, counts, fb, npix);
    else k_finalize_counts<<<blocks, 256, 0, st>>>(accum, counts, fb, npix);
    return cudaGetLastError();
}

cudaError_t launch_trace_rays_half(const RenderLaunch &p, bool octree, const uint2 *geom_h, const HalfPairs &hp, const float *org, const float *dir,
                                   int n, int *out_idx, float *out_t, cudaStream_t st) {
    h16::PairView pv;
    h16::NodeTab nt;
    half_views(hp, pv, nt);
    // whole blocks of whole warps: coop_trace_h is a full-warp collective
    const unsigned blocks = (unsigned)((n + kRenderThreads - 1) / kRenderThreads);
    if (octree) h16::k_trace_rays_h<true><<<blocks, kRenderThreads, 0, st>>>(p, geom_h, pv, nt, org, dir, n, out_idx, out_t);
    else h16::k_trace_rays_h<false><<<blocks, kRenderThreads, 0, st>>>(p, geom_h, pv, nt, org, dir, n, out_idx, out_t);
    return cudaGetLastError();
}
cudaError_t launch_camera_rays_half(const __half *cam_h, int n, const float *s, const float *t, uint32_t *states, float *org, float *dir,
                                    cudaStream_t st) {
    h16::k_camera_rays_h<<<(n + 127) / 128, 128, 0, st>>>(cam_h, n, s, t, states, org, dir);
    return cudaGetLastError();
}
cudaError_t launch_scatter_rays_half(const SceneView &sc, const uint2 *geom_h, const uint2 *matl_h, int n, const int *sphere_idx, const float *org,
                                     const float *dir, const float *t_hit, uint32_t *states, float *out_p, float *out_n, float *out_dir,
                                     float *out_att, int *scattered, cudaStream_t st) {
    h16::k_scatter_rays_h<<<(n + 127) / 128, 128, 0, st>>>(geom_h, matl_h, sc.tag, sc.n, n, sphere_idx, org, dir, t_hit, states, out_p, out_n,
                                                            out_dir, out_att, scattered);
    return cudaGetLastError();
}

// (re)build the pair lists of the USE_FP16 path: lists = 1 (flat mode) or kCells (octree mode)
cudaError_t build_half_pairs(HalfPairs &hp, const uint2 *geom_h, const int *tag, int n, bool octree, const TreeView &tv, cudaStream_t st) {
    const int lists = octree ? kCells : 1;
    cudaError_t e;
    if ((e = hp.count.reserve(kCells + 1)) != cudaSuccess || (e = hp.start.reserve(kCells + 2)) != cudaSuccess ||
        (e = hp.nodes.reserve(8 + 64 + 512)) != cudaSuccess || (e = hp.node_count.reserve(4 + 64 + 8)) != cudaSuccess)
        return e;
    if (octree) h16::k_fp16_nodes<<<1, 1, 0, st>>>(tv.cell_start, hp.nodes.ptr, hp.node_count.ptr);
    h16::k_pairs_count<<<(lists + 127) / 128, 128, 0, st>>>(tag, n, lists, tv.cell_start, tv.cell_list, tv.cell_cap, hp.count.ptr);
    h16::k_pairs_scan<<<1, 32, 0, st>>>(hp.count.ptr, lists, hp.start.ptr);
    uint32_t total = 0;
    if ((e = cudaMemcpyAsync(&total, hp.start.ptr + lists, 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
    hp.valid = false;                           // until the lists are rebuilt: a failure below must not leave stale lists marked usable
    if ((e = hp.geom.reserve((size_t)total + 1)) != cudaSuccess || (e = hp.idx.reserve((size_t)total + 1)) != cudaSuccess) return e;
    h16::k_pairs_fill<<<(lists + 127) / 128, 128, 0, st>>>(geom_h, tag, n, lists, tv.cell_start, tv.cell_list, tv.cell_cap, hp.start.ptr,
                                                           hp.geom.ptr, hp.idx.ptr);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    hp.pairs = total;
    hp.octree = octree;
    hp.valid = true;
    return cudaSuccess;
}

// Closest hit for caller-supplied rays (test hook: per-ray parity against the oracle's hitTree / hitable_list::hit)
__global__ void k_trace_rays(const __grid_constant__ RenderLaunch p, int octree, const float *__restrict__ org,
                             const float *__restrict__ dir, int n, int *__restrict__ out_idx, float *__restrict__ out_t) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const vec3f o = mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]), d = mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    TraceCounters tc;
    tc.sphere_tests = tc.node_tests = tc.voxel_steps = 0;
    const Hit h = octree ? trace_tree(p.scene, p.tree, &p.tree.planes[0][0], o, d, tc)
                         : trace_list(p.scene.geom, p.scene.tag, p.scene.n, o, d, tc);
    out_idx[i] = h.idx;
    out_t[i] = h.t;
}

// octree: the octree's grid, or the flat-list mode's grid over all spheres (p.tree); otherwise the N-test sweep
cudaError_t launch_trace_rays(const RenderLaunch &p, bool octree, const float *org, const float *dir, int n, int *out_idx,
                              float *out_t, cudaStream_t st) {
    const unsigned blocks = (unsigned)((n + kRenderThreads - 1) / kRenderThreads);
    // the render kernels' default trace: warp-cooperative (rt_coop.cuh) at p.coop_items candidates per lane; variant 1 = the per-lane walk
    if (octree && p.variant != 1 && p.coop_items == 4)
        coop::k_trace_rays_coop<4><<<blocks, kRenderThreads, 0, st>>>(p, org, dir, n, out_idx, out_t);
    else if (octree && p.variant != 1)
        coop::k_trace_rays_coop<2><<<blocks, kRenderThreads, 0, st>>>(p, org, dir, n, out_idx, out_t);
    else
        k_trace_rays<<<(n + 127) / 128, 128, 0, st>>>(p, octree ? 1 : 0, org, dir, n, out_idx, out_t);
    return cudaGetLastError();
}

// camera::get_ray (camera.h:45-49) and material::scatter (material.h:55-113) for caller-supplied inputs, evaluated by the same
// device functions the render kernels inline — the class-surface entry points of include/rt_dropin.h and a per-call parity hook.
__global__ void k_camera_rays(const CameraData cam, int n, const float *__restrict__ s, const float *__restrict__ t, uint32_t *__restrict__ states,
                              float *__restrict__ org, float *__restrict__ dir) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t *st = states + (size_t)i * 6;
    xorwow rng = xorwow_load(st);
    vec3f o, d;
    camera_ray(cam, s[i], t[i], rng, o, d);
    org[3 * i] = o.x; org[3 * i + 1] = o.y; org[3 * i + 2] = o.z;
    dir[3 * i] = d.x; dir[3 * i + 1] = d.y; dir[3 * i + 2] = d.z;
    xorwow_store(st, rng);
}
cudaError_t launch_camera_rays(const CameraData &cam, int n, const float *s, const float *t, uint32_t *states, float *org, float *dir,
                               cudaStream_t st) {
    k_camera_rays<<<(n + 127) / 128, 128, 0, st>>>(cam, n, s, t, states, org, dir);
    return cudaGetLastError();
}

// in: ray (org, dir), the sphere it hit and the ray parameter of the hit.  out: hit point = scattered origin, normal,
// scattered direction, attenuation, and whether the ray goes on (metal absorbs: material.h:72)
__global__ void k_scatter_rays(const SceneView sc, int n, const int *__restrict__ sphere_idx, const float *__restrict__ org,
                               const float *__restrict__ dir, const float *__restrict__ t_hit, uint32_t *__restrict__ states,
                               float *__restrict__ out_p, float *__restrict__ out_n, float *__restrict__ out_dir, float *__restrict__ out_att,
                               int *__restrict__ scattered) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int idx = sphere_idx[i];
    if (idx < 0 || idx >= sc.n || sc.tag[idx] < 0) { scattered[i] = -1; return; }
    uint32_t *st = states + (size_t)i * 6;
    xorwow rng = xorwow_load(st);
    const vec3f o = mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]), d = mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    vec3f hp, hn, att, dn = mk(0.f, 0.f, 0.f);
    hit_point(sc.geom[idx], o, d, t_hit[i], hp, hn);
    const bool go = scatter(sc.tag[idx], sc.matl[idx], d, hp, hn, att, dn, rng);
    out_p[3 * i] = hp.x; out_p[3 * i + 1] = hp.y; out_p[3 * i + 2] = hp.z;
    out_n[3 * i] = hn.x; out_n[3 * i + 1] = hn.y; out_n[3 * i + 2] = hn.z;
    out_dir[3 * i] = dn.x; out_dir[3 * i + 1] = dn.y; out_dir[3 * i + 2] = dn.z;
    out_att[3 * i] = att.x; out_att[3 * i + 1] = att.y; out_att[3 * i + 2] = att.z;
    scattered[i] = go ? 1 : 0;
    xorwow_store(st, rng);
}
cudaError_t launch_scatter_rays(const SceneView &sc, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                                uint32_t *states, float *out_p, float *out_n, float *out_dir, float *out_att, int *scattered, cudaStream_t st) {
    k_scatter_rays<<<(n + 127) / 128, 128, 0, st>>>(sc, n, sphere_idx, org, dir, t_hit, states, out_p, out_n, out_dir, out_att, scattered);
    return cudaGetLastError();
}

// fb = sqrt(accum * (1/ns)) (main.cu:111-114), for frames assembled from shards
__global__ void k_finalize(const float *__restrict__ accum, float *__restrict__ fb, size_t n3, float inv_ns) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n3) fb[i] = __fsqrt_rn(__fmul_rn(accum[i], inv_ns));
}

cudaError_t launch_finalize_n(const float *accum, float *fb, size_t n3, int ns, cudaStream_t st) {
    const float inv_ns = (float)(1.0 / (double)(float)ns);
    k_finalize<<<(unsigned)((n3 + 255) / 256), 256, 0, st>>>(accum, fb, n3, inv_ns);
    return cudaGetLastError();
}

cudaError_t launch_render(const RenderLaunch &p, bool octree, int sm_count, size_t smem_limit, cudaStream_t st,
                          int *blocks_out, int *kernel_out, int mode) {
    int dummy;
    int &which = kernel_out ? *kernel_out : dummy;
    const bool list = mode == kModeList, list_prog = mode == kModeListProgressive;
    // a pixel list gets the frame's choice, in its list (or list-progressive) instance
    if (octree) {
        // automatic choice by scene size (measured on B200, profiles/README.md r02f): the pixel-per-lane walk for small scenes
        // (short candidate lists, many empty voxels: C2 2.3 vs 3.4 ms), the warp-cooperative kernel from kCoopMinSpheres on
        // (C3 +8 %, C5 +19 % over the pooled kernel it replaced); variant 40 forces the cooperative kernel, variant 1 the per-lane walk
        if (p.variant == 40 || (p.variant != 1 && p.scene.n >= kCoopMinSpheres)) {
            which = kKernelCoop;
            // four candidates per lane once voxel lists are long (C5: 71 references per voxel, +4 %; C3: 13 per voxel, -6 %)
            auto kern = p.coop_items == 4 ? (list_prog ? coop::k_render_coop_pixels_progressive<4> : list ? coop::k_render_coop<4, true> : coop::k_render_coop<4>)
                                          : (list_prog ? coop::k_render_coop_pixels_progressive<2> : list ? coop::k_render_coop<2, true> : coop::k_render_coop<2>);
            return launch_persistent(kern, 0, p, sm_count, st, blocks_out, p);
        }
        which = kKernelLane;
        return launch_persistent(list_prog ? k_render_pixels_progressive<true, false> : list ? k_render<true, false, true> : k_render<true, false>, 0, p,
                                 sm_count, st, blocks_out, p);
    }
    which = kKernelListSweep;
    const size_t geom_bytes = (size_t)p.scene.n * sizeof(float4);
    if (geom_bytes + 1024 <= smem_limit)
        return launch_persistent(list_prog ? k_render_pixels_progressive<false, true> : list ? k_render<false, true, true> : k_render<false, true>,
                                 geom_bytes, p, sm_count, st, blocks_out, p);
    return launch_persistent(list_prog ? k_render_pixels_progressive<false, false> : list ? k_render<false, false, true> : k_render<false, false>, 0, p,
                             sm_count, st, blocks_out, p);
}

}  // namespace rt
