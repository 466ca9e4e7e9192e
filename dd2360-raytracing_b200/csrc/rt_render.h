// rt_render.h — launch interface of the persistent render kernel (rt_render.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "rt_types.h"

namespace rt {

constexpr int kRenderThreads = 128;
constexpr int kListGridMinSpheres = 256;   // flat-list mode: scenes at least this large are answered through the grid
constexpr int kCoopMinSpheres = 40000;   // octree mode: scenes at least this large use the warp-cooperative kernel (rt_coop.cuh)

struct RenderLaunch {
    SceneView scene;
    TreeView tree;
    alignas(16) CameraData cam;   // camera.h:51-58 as computed by k_camera_setup for THIS context and frame size (16-byte
                                  // aligned: the render kernels fetch it with 128-bit uniform loads from the constant bank)
    int nx, ny;
    int ns_total;            // samples per pixel of the whole frame (divisor of the final average)
    int ns_local;            // samples this launch traces per pixel
    int max_depth;
    int tiles_x;             // 8x4 pixel tiles per row
    int tile_first, tile_stride;   // this shard owns tiles tile_first + k*tile_stride
    uint32_t total_items;    // owned tiles * 32
    unsigned long long seed_offset;   // added to the per-pixel seed 1984 + pixel_index (spp shards)
    const uint32_t *seed_states;      // 6 words {d, v0..v4} per pixel to START from (RT_SEED_UPSTREAM: from k_seed_upstream; progressive
                                      // continuation: the states the previous call stored); nullptr = seed in the kernel (HEAD)
    union {
        uint32_t *state_out;          // progressive rendering (main.cu:119-142): every pixel's stream state is stored here when its
                                      // samples of this call are done (same layout); nullptr otherwise
        const uint32_t *pixels;       // pixel-list launches (rt_render_pixels, never progressive): item k renders pixel pixels[k]
                                      // into out[3k], seed_states then holds one state per entry.  Sharing the slot keeps the launch
                                      // parameters' size, so the parameters after them and the whole-frame instances' SASS stay put
    };
    int accumulate;                   // 1: a pixel's sum CONTINUES from the value in `out` (fb += col, main.cu:141, in one-shot order)
    int coop_items;          // cooperative kernel: candidates per lane and chunk step (2, or 4 for scenes with long voxel lists); 0 = 2
    int variant;             // kernel variant for A/B measurements (rt_render_args.tune[1]); 0 = default
    int finalize;            // 1: write sqrt(sum/ns) (main.cu:111-115); 0: write the linear sum
    float *out;              // nx*ny*3 floats (pixel lists: count*3, in list order)
    uint32_t *work_counter;  // queue head
    unsigned long long *counters;   // [0] rays, [1] paths
};

// which kernel a launch used (reported in rt_render_stats::kernel_id; names: rt_kernel_name)
enum KernelId { kKernelNone = 0, kKernelLane = 1, kKernelListSweep = 2, kKernelCoop = 4, kKernelHalf = 5 };
// list: p.pixels holds a pixel list (the LIST instance of the kernel the frame would use)
cudaError_t launch_render(const RenderLaunch &p, bool octree, int sm_count, size_t smem_limit, cudaStream_t st,
                          int *blocks_out, int *kernel_out, bool list = false);
cudaError_t launch_trace_rays(const RenderLaunch &p, bool octree, const float *org, const float *dir, int n, int *out_idx,
                              float *out_t, cudaStream_t st);
cudaError_t launch_camera_rays(const CameraData &cam, int n, const float *s, const float *t, uint32_t *states, float *org, float *dir,
                               cudaStream_t st);
cudaError_t launch_scatter_rays(const SceneView &sc, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                                uint32_t *states, float *out_p, float *out_n, float *out_dir, float *out_att, int *scattered, cudaStream_t st);
// render_init with the upstream seeding curand_init(1984, pixel_index + subsequence_base, 0) (main.cu:90)
cudaError_t launch_seed_upstream(uint32_t *states, size_t npix, unsigned long long seed, unsigned long long subsequence_base,
                                 const uint32_t *tables, cudaStream_t st);
// the same for a pixel list: states[k] = curand_init(seed, pixels[k], 0) for the entries < npix (the others are never read)
cudaError_t launch_seed_upstream_list(uint32_t *states, const uint32_t *pixels, int count, size_t npix, unsigned long long seed,
                                      const uint32_t *tables, cudaStream_t st);
// ---- USE_FP16 path (rt_render_half.cuh) ----
cudaError_t launch_scene_to_half(const float4 *geom, const float4 *matl, int n, uint2 *geom_h, uint2 *matl_h, cudaStream_t st);
cudaError_t launch_camera_setup_half(const float lookfrom[3], const float lookat[3], const float vup[3], float vfov, int nx, int ny,
                                     float aspect_override, float aperture, float focus_dist, __half *cam_h, cudaStream_t st);
struct HalfPairs {            // candidate lists as transposed sphere pairs (rt_half.cuh PairView), owned by the context
    uint4 *geom = nullptr;
    int2 *idx = nullptr;
    uint32_t *start = nullptr, *count = nullptr;
    uint2 *nodes = nullptr;          // compact per-level tables of the existing octree nodes (rt_half.cuh NodeTab)
    uint32_t *node_count = nullptr;
    size_t cap = 0;
    uint32_t pairs = 0;
    bool valid = false, octree = false;
};
cudaError_t build_half_pairs(HalfPairs &hp, const uint2 *geom_h, const int *tag, int n, bool octree, const TreeView &tv, cudaStream_t st);
cudaError_t launch_render_half(const RenderLaunch &p, bool octree, const uint2 *geom_h, const uint2 *matl_h, const __half *cam_h,
                               const HalfPairs &hp, int sm_count, cudaStream_t st, int *blocks_out, bool list = false);
// fb = the USE_FP16 build's sqrt(accum / ns) on `count` half sums widened to float
cudaError_t launch_finalize_half(const float *accum, float *fb, size_t count, int ns, cudaStream_t st);
// per-ray queries of the USE_FP16 build (hitTree / hitable_list::hit, camera::get_ray, material::scatter): float inputs are
// rounded to half, outputs are halves widened to float
cudaError_t launch_trace_rays_half(const RenderLaunch &p, bool octree, const uint2 *geom_h, const HalfPairs &hp, const float *org, const float *dir,
                                   int n, int *out_idx, float *out_t, cudaStream_t st);
cudaError_t launch_camera_rays_half(const __half *cam_h, int n, const float *s, const float *t, uint32_t *states, float *org, float *dir,
                                    cudaStream_t st);
cudaError_t launch_scatter_rays_half(const SceneView &sc, const uint2 *geom_h, const uint2 *matl_h, int n, const int *sphere_idx, const float *org,
                                     const float *dir, const float *t_hit, uint32_t *states, float *out_p, float *out_n, float *out_dir,
                                     float *out_att, int *scattered, cudaStream_t st);
// ---- output_to_stream on the device (rt_ppm.cu) ----
struct PpmWorkspace {
    uint32_t *block_len = nullptr;
    unsigned long long *block_off = nullptr;
    size_t block_cap = 0;
    char *text = nullptr;
    size_t text_cap = 0, text_len = 0;
};
cudaError_t ppm_format_device(PpmWorkspace &ws, const float *fb, int nx, int ny, cudaStream_t st, size_t *len_out);
void ppm_free(PpmWorkspace &ws);
cudaError_t launch_finalize(const float *accum, float *fb, int nx, int ny, int ns, cudaStream_t st);
cudaError_t launch_finalize_n(const float *accum, float *fb, size_t count, int ns, cudaStream_t st);

}  // namespace rt
