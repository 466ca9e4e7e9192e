/*
 * rt_abi.h — C ABI of librt_b200.so: the B200-native (sm_100a) render hot path of DD2360-RayTracing.
 *
 * The reference has no plugin / FFI layer: its "interface" for this path is the set of call sites in
 * main() (main.cu:347-477) plus the header class surface.  Every entry point below names the reference call
 * site it replaces.  Plain C: opaque handle, pointers and sizes only; no C++ types, no exceptions, no torch.
 * Every function returns 0 on success or a non-zero code (a cudaError_t value, or RT_ERR_* below) and leaves a
 * message retrievable with rt_last_error().  A context is bound to one GPU and one stream and is not
 * thread-safe (the reference is single-threaded on the default stream, main.cu:388-429).
 *
 * There is NO CPU fallback: if no CUDA device is usable rt_create fails.
 */
#ifndef RT_ABI_H
#define RT_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 1

enum {
    RT_OK = 0,
    RT_ERR_INVALID = 10001,      /* bad argument */
    RT_ERR_STATE = 10002,        /* call order: e.g. render before a scene exists */
    RT_ERR_UNSUPPORTED = 10003
};

/* material tags (material.h:52,62,76) */
enum { RT_MAT_NONE = -1, RT_MAT_LAMBERTIAN = 0, RT_MAT_METAL = 1, RT_MAT_DIELECTRIC = 2 };
/* per-pixel stream seeding: RT_SEED_HEAD = curand_init(1984 + pixel_index, 0, 0) (main.cu:93);
 * RT_SEED_UPSTREAM = curand_init(1984, pixel_index, 0) (main.cu:90, commented out in the reference) */
enum { RT_SEED_HEAD = 0, RT_SEED_UPSTREAM = 1 };
/* how a frame is split over ranks (SURVEY §8e): whole frame, interleaved pixel tiles (bit-identical to the
 * 1-GPU image after the sum), or samples-per-pixel shards (statistically equivalent, not bit-identical) */
enum { RT_SHARD_NONE = 0, RT_SHARD_TILES = 1, RT_SHARD_SPP = 2 };
/* arithmetic: RT_PREC_FP32 = the default build (real_t = float, precision_types.h:179); RT_PREC_FP16 = the reference
 * compiled with USE_FP16 (precision_types.h:8): real_t is a __half wrapper, the scene is the FP32 scene rounded to half,
 * frames are half values widened to float */
enum { RT_PREC_FP32 = 0, RT_PREC_FP16 = 1 };

/* One sphere and its material, flattened: what `sphere(center, radius, new <material>(...))` carries
 * (sphere.h:10, material.h:54,64,78).  36 bytes, same layout the oracle uses. */
typedef struct rt_sphere_desc {
    float cx, cy, cz, radius;
    int32_t mat;            /* RT_MAT_*; RT_MAT_NONE marks a slot create_world never wrote (never hit) */
    float ax, ay, az;       /* albedo: lambertian, metal */
    float param;            /* metal: fuzz (clamped to <= 1 as metal::metal does); dielectric: ref_idx */
} rt_sphere_desc;

/* camera(lookfrom, lookat, vup, vfov, aspect, aperture, focus_dist) — camera.h:22 */
typedef struct rt_camera_desc {
    float lookfrom[3], lookat[3], vup[3];
    float vfov, aspect, aperture, focus_dist;
} rt_camera_desc;

typedef struct rt_octree_stats {
    int32_t node_count, leaf_count;     /* Octree::nodeCount / leafCount */
    int64_t entries;                    /* (cell, sphere) entries stored in leaf buckets */
    int64_t dropped_full;               /* entries the reference drops with "Leaf nodes full" */
    int64_t dropped_outside;            /* spheres outside the root box */
    int64_t fine_voxels, fine_refs;     /* internal sub-grid size (not part of the reference layout) */
    float build_ms;                     /* device time of the whole build */
} rt_octree_stats;

typedef struct rt_render_args {
    int32_t nx, ny;          /* image size (main.cu:348-349) */
    int32_t ns;              /* samples per pixel of the WHOLE frame (main.cu:350) */
    int32_t max_depth;       /* 50 (main.cu:47); 0 selects 50 */
    int32_t use_octree;      /* USE_OCTREE (main.cu:24): 1 = hitTree, 0 = hitable_list::hit */
    int32_t seed_mode;       /* RT_SEED_* */
    int32_t shard_mode;      /* RT_SHARD_* */
    int32_t shard_rank, shard_count;
    int32_t precision;       /* RT_PREC_* (USE_FP16, precision_types.h:8); FP16 shards by tiles only (RT_SHARD_TILES: the summed
                              * half sums are the 1-GPU sums exactly; finalise them with rt_finalize_ex(.., RT_PREC_FP16)) */
    int32_t tune[6];         /* kernel A/B knobs for measurements and tests; 0 = defaults; they never change the image.
                              * [1] kernel variant: 0 automatic, 1 pixel-per-lane kernel (and per-lane rt_trace_rays), 20 flat
                              * list as an N-test sweep, 31 single-pixel queue, 40 warp-cooperative kernel; other values select
                              * the automatic choice.  [0], [2..5] reserved (ignored) */
} rt_render_args;

typedef struct rt_render_stats {
    uint64_t rays;           /* closest-hit queries = iterations of color()'s loop (main.cu:47) */
    uint64_t paths;          /* camera samples */
    uint64_t sphere_tests;   /* ray-sphere tests executed (only counted when built with RT_COUNTERS) */
    uint64_t node_tests;     /* octree node tests executed (same) */
    float kernel_ms;         /* device time of the render kernel(s), CUDA events on the context's stream */
    int32_t launches;        /* kernels launched by this call */
    int32_t kernel_id;       /* which render kernel ran (rt_kernel_name) */
    int32_t reserved;
} rt_render_stats;

typedef struct rt_context rt_context;

/* ---- context ---------------------------------------------------------------------------------------- */
int rt_abi_version(void);
int rt_create(int device, rt_context **out);                 /* replaces nothing; cudaSetDevice + stream */
void rt_destroy(rt_context *ctx);                            /* replaces free_world + cudaFree x7 (main.cu:459-474) */
const char *rt_last_error(const rt_context *ctx);
/* cudaStream_t to launch on.  NULL = the context's own stream (a BLOCKING stream: ordered with the legacy default stream).
 * To run on the legacy default stream itself pass cudaStreamLegacy ((void *)0x1), not NULL. */
int rt_set_stream(rt_context *ctx, void *cuda_stream);
const char *rt_kernel_name(int kernel_id);                   /* name of rt_render_stats::kernel_id */
int rt_device_info(const rt_context *ctx, int *sm_count, int *clock_khz, size_t *mem_bytes);

/* ---- scene: replaces rand_init + create_world (main.cu:388,399) ------------------------------------------ */
/* The reference's generator: world seed 1984, NUM_SPHERES = n, SPHERE_RADIUS = radius (main.cu:22-23,146-181). */
int rt_scene_generate(rt_context *ctx, int n, float sphere_radius);
/* same under a given arithmetic: with RT_PREC_FP16 every value is stored through real_t (rounded to half) and the material
 * choice compares a half-rounded draw with half-rounded thresholds, which changes the draw sequence (main.cu:165-172) */
int rt_scene_generate_ex(rt_context *ctx, int n, float sphere_radius, int precision);
/* A caller-built world (the drop-in headers flatten hitable_list into this). */
int rt_scene_upload(rt_context *ctx, const rt_sphere_desc *spheres, int n);
int rt_scene_download(rt_context *ctx, rt_sphere_desc *out, int n);
int rt_scene_size(const rt_context *ctx);
/* camera: main.cu:192-202 constants with aspect = nx/ny when desc == NULL */
int rt_camera_set(rt_context *ctx, const rt_camera_desc *desc, int nx, int ny);
int rt_camera_get(rt_context *ctx, float out22[22]);         /* origin,llc,horizontal,vertical,u,v,w,lens_radius */
/* the camera the USE_FP16 build constructs for an nx x ny frame (half values widened to float) */
int rt_camera_get_half(rt_context *ctx, int nx, int ny, float out22[22]);

/* ---- octree: replaces D2H(spheres) + buildOctree + H2D(Octree) (main.cu:405-415) -------------------------- */
int rt_octree_build(rt_context *ctx, int spheres_per_leaf, rt_octree_stats *stats);
/* same for a given arithmetic: with RT_PREC_FP16 `intersects` (acceleration_structure.h:82-93) compares half-rounded
 * centres against half-rounded grown bounds, which moves spheres between cells */
int rt_octree_build_ex(rt_context *ctx, int spheres_per_leaf, int precision, rt_octree_stats *stats);
size_t rt_octree_reference_bytes(int spheres_per_leaf);      /* sizeof(Octree) for that SPHERES_PER_LEAF */
/* sizeof(Octree) of the build with that arithmetic: RT_PREC_FP32 is rt_octree_reference_bytes; under RT_PREC_FP16 the AABB
 * holds six halves, so an OctNode is 48 bytes instead of 60 (OctLeaf and the two counts are ints in both).  0 for an unknown
 * precision or spheres_per_leaf < 1.  Needs no GPU. */
size_t rt_octree_reference_bytes_ex(int spheres_per_leaf, int precision);
/* the tree in the reference's own memory layout (acceleration_structure.h:23-61), for the bit-exact check.  A tree built with
 * RT_PREC_FP16 comes out in the layout of the USE_FP16 build (rt_octree_reference_bytes_ex(.., RT_PREC_FP16) bytes): the box
 * planes are exact in half, so its AABBs are the FP32 build's rounded to half; its buckets hold the FP16 build's memberships. */
int rt_octree_export_reference(rt_context *ctx, void *host_blob, size_t bytes);

/* test hook: read one internal traversal array back (0 grid descriptor, 1 voxel records, 2 voxel references,
 * 3 per-sphere entry offsets, 4 per-sphere cell lists, 5 big-sphere list, 6 sphere flags, 7 per-cell list offsets (513),
 * 8 per-cell sphere lists in Morton cell order).  Returns the byte size
 * (host == NULL) or bytes copied. */
size_t rt_octree_debug_read(rt_context *ctx, int which, void *host, size_t cap);

/* cuRAND XORWOW state {d, v0..v4} after curand_init(seed, subsequence, 0) (curand_kernel.h:772-797), evaluated on the host
 * with the skip-ahead matrices this library derives itself; subsequence < 2^40.  What RT_SEED_UPSTREAM gives pixel
 * `subsequence` (seed 1984, main.cu:90).  Needs no GPU. */
int rt_xorwow_state(unsigned long long seed, unsigned long long subsequence, uint32_t out6[6]);

/* test hook: raw device counters of the last render call.  [0] rays, [1] paths; RT_COUNTERS builds add [2] sphere tests,
 * [3] visibility line tests and [4] voxel steps. */
int rt_debug_counters(rt_context *ctx, uint64_t out[32]);

/* test hook: closest hit (sphere index or -1, and t) of n caller-supplied rays — hitTree / hitable_list::hit per ray, answered by
 * the walk the FP32 render kernels use for the same scene, so that each of them can be held to a reference ray by ray:
 *   octree            : the warp-cooperative walk (two candidates per lane, four once voxel lists average 40 or more references);
 *   flat list         : below 256 spheres the N-test sweep; from 256 on the same walks over the grid of all spheres the render
 *                       builds for that mode (built here on first use);
 * the environment variable RT_RENDER_VARIANT, read by rt_create, selects another walk: 1 the per-lane grid walk, 20 the N-test
 * sweep (flat list), 40 the cooperative walk.  Every walk returns the same index and t.  Outside the contract (the answer may differ
 * from the reference's): in octree mode, a zero direction component with the origin exactly on one of the reference's level-3 cell
 * planes of that axis (x, z = -11 + 2.75k, y = 0.25k), where the reference's own slab test divides 0 by 0.  An octree query on a tree built for RT_PREC_FP16 is RT_ERR_STATE
 * ("other precision"), as in rt_trace_rays_ex. */
int rt_trace_rays(rt_context *ctx, int use_octree, int n, const float *org, const float *dir, int *out_idx, float *out_t);

/* camera::get_ray(s, t, &rand_state) (camera.h:45-49) for n (s, t) pairs, each drawing its lens sample from its own XORWOW
 * state (6 words {d, v0..v4}, host array, updated in place; start one with rt_xorwow_state); org / dir: 3 floats per ray.
 * Evaluated on the GPU by the device function the render kernels inline. */
int rt_camera_get_rays(rt_context *ctx, int n, const float *s, const float *t, uint32_t *states6, float *org, float *dir);
/* material::scatter (material.h:55-113) with the hit record sphere::hit fills (sphere.h:30-33), for n (ray, sphere, t):
 * out_p = hit point = origin of the scattered ray, out_normal, out_dir = scattered direction, out_atten = attenuation,
 * scattered = 1 / 0 (metal absorbs, material.h:72) / -1 (not a defined sphere).  States as in rt_camera_get_rays. */
int rt_scatter_rays(rt_context *ctx, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                    uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten, int *scattered);

/* The three queries above under a given arithmetic.  RT_PREC_FP32: exactly rt_trace_rays / rt_camera_get_rays / rt_scatter_rays.
 * RT_PREC_FP16: what the reference's USE_FP16 build computes, by the device functions the FP16 render composes — every float
 * input is rounded to half (nearest) on entry and every output is a half widened to float, so outputs go back in exactly.
 *   rt_trace_rays_ex      hitTree (octree: ground sphere first, then the stored list of every level-3 cell whose half AABB the
 *                         ray's line crosses) or hitable_list::hit over every sphere; out_t = +inf on a miss (FLT_MAX in half)
 *   rt_camera_get_rays_ex camera::get_ray with the half camera of the frame size of the last rt_camera_set (rt_camera_get_half)
 *   rt_scatter_rays_ex    sphere::hit's hit record (p, normal) from the half t, then material::scatter, all in half
 * Errors: unknown precision -> RT_ERR_INVALID; no scene (trace, scatter), no camera (camera), no octree, or an octree query in
 * one precision on a tree built for the other (rt_octree_build_ex) -> RT_ERR_STATE. */
int rt_trace_rays_ex(rt_context *ctx, int use_octree, int precision, int n, const float *org, const float *dir, int *out_idx, float *out_t);
int rt_camera_get_rays_ex(rt_context *ctx, int precision, int n, const float *s, const float *t, uint32_t *states6, float *org, float *dir);
int rt_scatter_rays_ex(rt_context *ctx, int precision, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                       uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten, int *scattered);

/* ---- render: replaces render_init + render (main.cu:424-429) ---------------------------------------------- */
/* Renders this rank's shard into `accum_dev` (device pointer, nx*ny*3 floats): LINEAR radiance sums (before
 * /ns and sqrt), zero where the shard owns nothing, so that shards add up (main.cu:119-142 semantics). */
int rt_render_accumulate(rt_context *ctx, const rt_render_args *args, float *accum_dev, rt_render_stats *stats);
/* Progressive rendering — render_progressive (main.cu:119-142) with its state carry: every call traces args->ns MORE samples
 * per pixel, resuming each pixel's XORWOW stream where the previous call stored it (rng_state_dev: 6 words {d, v0..v4} per
 * pixel, nx*ny*24 bytes of device memory owned by the caller; main.cu:136) and continuing each pixel's sum from the value
 * in accum_dev in the order a one-shot render adds its samples (main.cu:141).  k calls of m samples therefore leave, bit for
 * bit, the linear sums (and stream states) of one k*m-sample rt_render_accumulate.  first != 0 starts the streams
 * (args->seed_mode) and overwrites accum_dev.  Dump a frame at any point with rt_finalize(.., samples so far).  Under
 * RT_PREC_FP16 each pixel's sum is the half accumulator of the reference's FP16 build (widened to float, resumed exactly); dump
 * with rt_finalize_ex(.., samples so far, RT_PREC_FP16).  Tile shards (RT_SHARD_TILES) may render progressively too. */
int rt_render_progressive(rt_context *ctx, const rt_render_args *args, float *accum_dev, uint32_t *rng_state_dev, int first,
                          rt_render_stats *stats);
/* statistics of the last rt_render* call made with stats == NULL (the call then returns without waiting for the kernel, so a
 * collective or a copy can be queued right behind it); waits for the context's stream */
int rt_last_render_stats(rt_context *ctx, rt_render_stats *stats);
/* fb = sqrt(accum * (1/ns)) per channel (main.cu:111-114); in place allowed */
int rt_finalize(rt_context *ctx, const float *accum_dev, float *fb_dev, int nx, int ny, int ns);
/* the same on `count` consecutive floats: a rank's slice of the frame after rt_reduce_scatter */
int rt_finalize_n(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns);
/* the same for a given arithmetic: RT_PREC_FP32 is rt_finalize_n; RT_PREC_FP16 reads half sums widened to float and computes
 * what the FP16 build's render does (main.cu:111-115): col * real_t(1.0 / real_t(ns)) in half, sqrt in float, rounded to half.
 * In place allowed; an unknown precision or ns < 1 is RT_ERR_INVALID. */
int rt_finalize_ex(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns, int precision);
/* Whole frame on one GPU straight into the reference's fb layout (device pointer, vec3 per pixel). */
int rt_render(rt_context *ctx, const rt_render_args *args, float *fb_dev, rt_render_stats *stats);
/* Same with a HOST destination: render + device->host copy (what the reference does through managed memory). */
int rt_render_to_host(rt_context *ctx, const rt_render_args *args, float *fb_host, rt_render_stats *stats);
/* Render only the pixels listed in pixels_dev (device memory: count uint32 pixel indices j*nx + i of the args->nx x args->ny
 * frame, any order, duplicates allowed).  out_dev (device memory) receives count*3 floats in LIST order: entry k holds exactly
 * what rt_render (finalize != 0) or rt_render_accumulate (finalize == 0) writes for pixel pixels_dev[k] of the same frame with
 * the same args, bit for bit, in either precision and seeding.  An entry >= nx*ny yields (0, 0, 0) and traces nothing.
 * Every pixel's result depends only on its own stream and sample chain, so a crop, a region or a few pixels of interest cost
 * what their own rays cost.  The kernel is chosen as for the frame (from the scene and args->tune[1], not from count);
 * RT_SEED_UPSTREAM seeds the listed pixels only (count x 24 bytes).  Stats as for frames: rays summed over the entries,
 * paths = ns x the in-range entries.  A null pointer, count < 1, args->shard_mode != RT_SHARD_NONE, or a pixels_dev / out_dev
 * that is not device (or managed) memory of the context's GPU -> RT_ERR_INVALID; no scene, or an octree built for the other
 * precision -> RT_ERR_STATE; nothing is written on an error.  The list is rendered in the order given: list neighbouring
 * pixels next to each other (e.g. in 8x4 tiles, as the frame queue does) for coherent warps. */
int rt_render_pixels(rt_context *ctx, const rt_render_args *args, const uint32_t *pixels_dev, int count, float *out_dev,
                     int finalize, rt_render_stats *stats);
/* Progressive rendering of the pixels listed in pixels_dev (device memory: count uint32 pixel indices j*nx + i).  accum_dev
 * (nx*ny*3 floats) and rng_state_dev (nx*ny*6 words) are FRAME-indexed: the very buffers rt_render_progressive uses, so the
 * two calls interleave freely.  Each distinct listed pixel gets args->ns MORE samples: its stream resumes from
 * rng_state_dev[6*pix] and its sum continues from accum_dev[3*pix] (first == 0), or its stream is started with
 * args->seed_mode and its sum overwritten (first != 0).  A pixel listed more than once in a call is rendered once.  Entries
 * >= nx*ny and pixels not listed are left untouched in all three buffers.  counts_dev (optional, nx*ny uint32): counts[pix]
 * += args->ns for every rendered pixel (= args->ns when first != 0).  Any schedule of rt_render_progressive and
 * rt_render_pixels_progressive calls that gives a pixel S samples in total leaves its sum and state bit-identical to a
 * one-shot S-sample render of that pixel (rt_render_accumulate / rt_render_progressive(first=1)), in either precision and
 * seeding.  rt_render_progressive takes no counts: a caller that mixes the two adds the frame call's ns to every pixel's
 * count.  The kernel is chosen as for the frame; shards are refused; stats as rt_render_pixels (paths = ns x rendered
 * pixels); stats == NULL is asynchronous (rt_last_render_stats).  A null args / pixels_dev / accum_dev / rng_state_dev,
 * count < 1, bad nx/ny/ns, args->shard_mode != RT_SHARD_NONE, an unknown seed mode or precision, or a given pointer (counts_dev
 * included) that is not device (or managed) memory of the context's GPU -> RT_ERR_INVALID; no scene, USE_OCTREE without an
 * octree, or an octree built for the other precision -> RT_ERR_STATE; nothing is written on an error. */
int rt_render_pixels_progressive(rt_context *ctx, const rt_render_args *args, const uint32_t *pixels_dev, int count,
                                 float *accum_dev, uint32_t *rng_state_dev, uint32_t *counts_dev, int first,
                                 rt_render_stats *stats);
/* fb = what rt_render writes for a pixel rendered with counts[pix] samples: sqrt(sum * (1/counts[pix])) per channel in the
 * given precision (RT_PREC_FP16: the USE_FP16 build's finalise, as rt_finalize_ex); counts[pix] == 0 gives (0, 0, 0).
 * npix pixels (3*npix floats), in place allowed.  A null pointer, a pointer that is not device (or managed) memory of the
 * context's GPU, or an unknown precision -> RT_ERR_INVALID. */
int rt_finalize_counts(rt_context *ctx, const float *accum_dev, const uint32_t *counts_dev, float *fb_dev, size_t npix,
                       int precision);

/* Adaptive sampling: each 8x4 tile of the frame queue gets as many samples as its noise estimate asks for, between
 * params->min_spp and args->ns (= max_spp, the per-pixel budget, in [min_spp, 65536]).  The estimate of a pixel compares two
 * independent segments of its own sample chain, [0, a) and [a, c), in display space, scaled to the standard error of its c-sample
 * mean (e_p, rt_adaptive.h); a tile's error E_t is the largest e_p of its in-frame pixels (NaN counts as +inf).  The call
 *   1. renders the whole frame progressively with min_spp/2 samples (first = 1), snapshots the sums, renders min_spp/2 more, and
 *      sets counts := min_spp;
 *   2. runs rounds: every tile not yet done with c < max_spp and !(E_t <= threshold) takes its sums as its new snapshot and gets
 *      min(c, max_spp - c) more samples (one rt_render_pixels_progressive call over those tiles, in tile order); any other tile
 *      is done and never evaluated again.  The rounds end when a selection lists nothing (at most ceil(log2(max/min)));
 *   3. finalises the frame from the counts into fb_dev (rt_finalize_counts).
 * accum_dev (nx*ny*3 floats), rng_state_dev (nx*ny*6 words) and counts_dev (nx*ny uint32) are the frame-indexed buffers of
 * rt_render_progressive and rt_render_pixels_progressive, so a caller may keep refining with those.  Every pixel ends, bit for
 * bit, where rt_render(ns = counts[pix]) puts it (fb), and its sum and state where a one-shot counts[pix]-sample progressive render
 * does, in either precision and seeding.  err_dev (optional, nx*ny floats): e_p of every pixel from its last two segments.
 * threshold = +inf gives a uniform min_spp frame.  stats (optional): rays, paths and test counters summed over the render calls,
 * their launches, the render kernel's id, kernel_ms = device time of the whole call, the rounds and the pixels listed in each.  The
 * call waits for the stream once per round (the list length is read back).  A null args / params / accum_dev / rng_state_dev /
 * counts_dev / fb_dev, bad nx/ny, an odd min_spp or min_spp < 2, max_spp out of range, a NaN or negative threshold,
 * args->shard_mode != RT_SHARD_NONE, an unknown seed mode or precision, or a given pointer that is not device (or managed) memory
 * of the context's GPU -> RT_ERR_INVALID; no scene, USE_OCTREE without an octree, or an octree built for the other precision ->
 * RT_ERR_STATE; nothing is written on an error. */
typedef struct rt_adaptive_params {
    int32_t min_spp;        /* even, >= 2: two whole-frame segments of min_spp/2 give the first estimate */
    float threshold;        /* display-space standard error a tile must reach; +inf = uniform min_spp frame */
    int32_t reserved[6];
} rt_adaptive_params;
typedef struct rt_adaptive_stats {
    rt_render_stats render; /* rays/paths summed over all calls; kernel_ms spans the whole call; kernel_id of the render kernel */
    int32_t rounds, reserved;
    uint64_t round_pixels[16];   /* pixels listed in round r */
} rt_adaptive_stats;
int rt_render_adaptive(rt_context *ctx, const rt_render_args *args, const rt_adaptive_params *params, float *accum_dev,
                       uint32_t *rng_state_dev, uint32_t *counts_dev, float *fb_dev, float *err_dev, rt_adaptive_stats *stats);

/* ---- output: replaces output_to_stream (main.cu:321-333) -------------------------------------------------- */
/* P3 text, byte-identical to the reference writer.  Returns bytes needed when buf == NULL. */
size_t rt_format_ppm(const float *fb_host, int nx, int ny, char *buf, size_t cap);
/* The same writer on the device (csrc/rt_ppm.cu): quantise + format in HBM, so only the text crosses PCIe — at 4K the host
 * writer above costs more than the render.  rt_ppm_format formats a DEVICE frame into a context-owned device buffer and
 * returns the text length; rt_ppm_read copies that text to the host (cap >= length).  rt_render_to_ppm = rt_render into
 * the context's scratch frame + rt_ppm_format: what main() does for output modes 0 and 3 (main.cu:427 + :435-452).
 * Bytes identical to rt_format_ppm for every finite frame. */
int rt_ppm_format(rt_context *ctx, const float *fb_dev, int nx, int ny, size_t *len_out);
int rt_ppm_read(rt_context *ctx, char *buf_host, size_t cap);
int rt_render_to_ppm(rt_context *ctx, const rt_render_args *args, rt_render_stats *stats, size_t *len_out);

/* ---- multi-GPU: one context per GPU, NCCL over NVLink ---------------------------------------------------------
 * The reference is single-GPU; this wraps the one exchange a sharded frame needs, between render (main.cu:427) and the
 * output switch (main.cu:435-453): the ranks' LINEAR radiance buffers (rt_render_accumulate with RT_SHARD_TILES or
 * RT_SHARD_SPP) are summed, then /ns, sqrt and the PPM writer run on the sum.  All calls are asynchronous on the context's
 * stream.  NCCL is looked up at run time (libnccl.so.2); without it these entry points return RT_ERR_UNSUPPORTED.
 *   one process per GPU : rank 0 calls rt_comm_get_unique_id, ships the 128 bytes to the others, all call rt_comm_init_rank;
 *   one process, n GPUs : rt_comm_init_all over n contexts, and collectives bracketed by rt_group_start / rt_group_end;
 *   caller-owned NCCL   : rt_comm_attach(ctx, ncclComm_t, nranks, rank). */
#define RT_COMM_ID_BYTES 128
int rt_comm_get_unique_id(void *id_out);
int rt_comm_init_rank(rt_context *ctx, const void *id, int nranks, int rank);
int rt_comm_init_all(rt_context *const *ctxs, int n);
int rt_comm_attach(rt_context *ctx, void *nccl_comm, int nranks, int rank);
int rt_comm_destroy(rt_context *ctx);
int rt_comm_rank(const rt_context *ctx);
int rt_comm_size(const rt_context *ctx);
int rt_group_start(void);
int rt_group_end(void);
/* sum of `count` floats over the ranks, in place, result on `root` */
int rt_reduce(rt_context *ctx, float *accum_dev, size_t count, int root);
/* sum over the ranks of accum_dev[nranks * slice_count]; rank r receives elements [r * slice_count, (r+1) * slice_count) —
 * every rank then finalises (and formats, and copies out) its own slice of the frame in parallel */
int rt_reduce_scatter(rt_context *ctx, const float *accum_dev, float *slice_dev, size_t slice_count);
int rt_broadcast(rt_context *ctx, void *dev, size_t bytes, int root);

/* ---- measurement: dense FP32 FFMA rate of this GPU (2 flop per FFMA), the denominator of the FP32 roofline -------- */
int rt_ffma_peak(rt_context *ctx, float *tflops, float *kernel_ms);
int rt_hfma2_peak(rt_context *ctx, float *tflops, float *kernel_ms);    /* packed half: 4 flop per HFMA2 (USE_FP16 roofline) */

/* ---- device memory helpers for hosts without a CUDA runtime binding ---------------------------------------- */
int rt_malloc(rt_context *ctx, size_t bytes, void **dev_ptr);
int rt_free(rt_context *ctx, void *dev_ptr);
int rt_memcpy_to_host(rt_context *ctx, void *host, const void *dev, size_t bytes);
int rt_synchronize(rt_context *ctx);

#ifdef __cplusplus
}
#endif
#endif
