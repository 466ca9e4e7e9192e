// rt_abi.cu — implementation of the C ABI in include/rt_abi.h (context, scene, camera, build, render, output).
// There is no CPU fallback anywhere in this library: every compute entry point launches CUDA kernels.
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <nccl.h>          // types and prototypes only: the functions are resolved with dlopen (see NcclApi)
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/rt_abi.h"
#include "rt_math.cuh"
#include "rt_adaptive.h"
#include "rt_build.cuh"
#include "rt_octree.h"
#include "rt_render.h"
#include "rt_xorwow_skip.h"

using namespace rt;

struct rt_context {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaDeviceProp prop{};
    std::string err;
    // scene
    int n = 0;
    Buffer<float4> geom, matl;
    Buffer<int> tag;
    // camera
    bool have_camera = false;
    int cam_nx = 0, cam_ny = 0;
    Buffer<CameraData> cam_dev;
    CameraData cam_host{};
    // octree
    OctreeBuilder octree;
    OctreeBuilder list_accel;      // USE_OCTREE off: the same grid over ALL spheres answers hitable_list::hit
    bool list_accel_valid = false;
    float grid_density = 4.0f;
    int default_variant = 0;       // RT_RENDER_VARIANT: kernel A/B override for whole test runs (0 = automatic)
    int last_kernel = 0;           // KernelId of the last render launch
    int last_launches = 0;         // kernels the last render call launched (upstream seeding + render)
    // render scratch
    Buffer<uint32_t> work_counter;
    Buffer<unsigned long long> counters;
    Buffer<float> scratch_fb;
    PpmWorkspace ppm;
    Buffer<char, Mem::Pinned> pinned;   // page-locked staging for the scene descriptors
    Buffer<char> desc_dev;              // ... and their raw device copy (split into geom / matl / tag by k_split_scene)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // RT_SEED_UPSTREAM: skip-ahead matrices (device copy) and the per-pixel stream states
    // RT_PREC_FP16: the scene rounded to half (8 B geometry + 8 B material per sphere) and the half camera
    Buffer<uint2> geom_h, matl_h;
    bool half_valid = false;
    HalfPairs half_pairs;
    Buffer<__half> cam_h;
    int cam_h_nx = 0, cam_h_ny = 0;
    rt_camera_desc cam_desc{};
    bool cam_desc_custom = false;
    Buffer<uint32_t> skip_tables;
    Buffer<uint32_t> seed_states;
    // rt_render_pixels_progressive: the deduplicated pixel list and the one-bit-per-frame-pixel mask that dedupes it
    Buffer<uint32_t> list_dedup, list_mask;
    // rt_render_adaptive: the snapshot sums (3 floats per pixel), the per-tile words of the selection pass (listed, offset, done),
    // its pixel list, the scan's temporary storage, and the events that bracket the whole call
    Buffer<float> ad_snap;
    Buffer<uint32_t> ad_tiles, ad_list, ad_scan;
    cudaEvent_t ad_ev0 = nullptr, ad_ev1 = nullptr;
    // multi-GPU (rt_comm_*): this context's rank in an NCCL communicator
    ncclComm_t comm = nullptr;
    bool comm_owned = false;
    int comm_rank = 0, comm_size = 1;
};

extern "C" int rt_comm_destroy(rt_context *ctx);

static const std::vector<uint32_t> &host_skip_tables() {
    static const std::vector<uint32_t> t = make_skip_tables();      // derived once per process (a few ms)
    return t;
}

static int fail(rt_context *ctx, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}
static int cuda_fail(rt_context *ctx, cudaError_t e, const char *what) {
    return fail(ctx, (int)e, "CUDA error = %u at %s '%s'", (unsigned)e, what, cudaGetErrorString(e));
}
#define CK(call)                                              \
    do {                                                      \
        cudaError_t e_ = (call);                              \
        if (e_ != cudaSuccess) return cuda_fail(ctx, e_, #call); \
    } while (0)

extern "C" int rt_abi_version(void) { return RT_ABI_VERSION; }

extern "C" int rt_create(int device, rt_context **out) {
    if (!out) return RT_ERR_INVALID;
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0) return e != cudaSuccess ? (int)e : (int)cudaErrorNoDevice;   // no CPU fallback
    if (device < 0 || device >= count) return RT_ERR_INVALID;
    rt_context *ctx = new rt_context();
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&ctx->prop, device)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamDefault)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ev1)) != cudaSuccess ||
        (e = cudaEventCreate(&ctx->ad_ev0)) != cudaSuccess || (e = cudaEventCreate(&ctx->ad_ev1)) != cudaSuccess ||
        (e = ctx->work_counter.reserve(1)) != cudaSuccess || (e = ctx->counters.reserve(32)) != cudaSuccess ||
        (e = ctx->cam_dev.reserve(1)) != cudaSuccess) {
        rt_destroy(ctx);
        return (int)e;
    }
    ctx->stream = ctx->own_stream;
    const char *dens = getenv("RT_GRID_DENSITY");
    if (dens && atof(dens) > 0) ctx->grid_density = (float)atof(dens);
    float flat = 0, wide = 0;
    unsigned flat_min = kFlatVoxelMinSpheres;
    const char *shape = getenv("RT_GRID_SHAPE");        // "flat:wide[:from how many spheres]", e.g. "1:1" for cubes everywhere
    if (shape && sscanf(shape, "%f:%f:%u", &flat, &wide, &flat_min) >= 2 && flat > 0 && wide > 0) {
        ctx->octree.grid_flat = ctx->list_accel.grid_flat = flat;
        ctx->octree.grid_wide = ctx->list_accel.grid_wide = wide;
        ctx->octree.grid_flat_min = ctx->list_accel.grid_flat_min = flat_min;
    }
    const char *var = getenv("RT_RENDER_VARIANT");
    if (var) ctx->default_variant = atoi(var);
    *out = ctx;
    return RT_OK;
}

// Also the failure path of rt_create, which may leave any of these unset.  The context's buffers free themselves.
extern "C" void rt_destroy(rt_context *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (cudaEvent_t ev : {ctx->ev0, ctx->ev1, ctx->ad_ev0, ctx->ad_ev1})
        if (ev) cudaEventDestroy(ev);
    rt_comm_destroy(ctx);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
}

extern "C" const char *rt_last_error(const rt_context *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

extern "C" int rt_set_stream(rt_context *ctx, void *s) {
    if (!ctx) return RT_ERR_INVALID;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return RT_OK;
}

extern "C" const char *rt_kernel_name(int kernel_id) {
    switch (kernel_id) {
        case kKernelLane: return "k_render<octree> (pixel per lane, grid walk)";
        case kKernelListSweep: return "k_render<list> (N-test sweep)";
        case kKernelCoop: return "k_render_coop (warp-cooperative candidate tests)";
        case kKernelHalf: return "k_render_h (USE_FP16)";
        default: return "none";
    }
}

extern "C" int rt_device_info(const rt_context *ctx, int *sm_count, int *clock_khz, size_t *mem_bytes) {
    if (!ctx) return RT_ERR_INVALID;
    if (sm_count) *sm_count = ctx->prop.multiProcessorCount;
    if (clock_khz) *clock_khz = ctx->prop.clockRate;
    if (mem_bytes) *mem_bytes = ctx->prop.totalGlobalMem;
    return RT_OK;
}

// ---- scene ------------------------------------------------------------------------------------------------------
// main.cu:146-181.  The generator is one sequential XORWOW stream (seed 1984, curand_init(1984,0,0), main.cu:80),
// so it runs on the host and the result is uploaded as SoA; arguments are drawn left to right as the device
// evaluates them (SURVEY D4).  No device heap, no per-sphere `new`.
static inline float round_half(float x) { return __half2float(__float2half_rn(x)); }

// fp16: the USE_FP16 build of create_world.  Every stored value goes through real_t(float|double), i.e. is rounded to
// half; the one place where that changes the CONTROL flow is `const real_t choose_mat = RND` compared with
// real_t(0.8f) / real_t(0.95f) (main.cu:165,168,172): a draw within half an ulp of a threshold picks another material,
// which consumes a different number of draws and shifts every later sphere.
static void generate_world(int n, float radius, bool fp16, std::vector<rt_sphere_desc> &out) {
    out.assign((size_t)n, rt_sphere_desc{0, 0, 0, 0, RT_MAT_NONE, 0, 0, 0, 0});
    if (n < 4) return;
    xorwow rng;
    xorwow_seed(rng, 1984ull);
    auto RND = [&]() { return xorwow_uniform(rng); };
    out[0] = rt_sphere_desc{0.f, -1000.f, -1.f, 1000.f, RT_MAT_LAMBERTIAN, 0.5f, 0.5f, 0.5f, 0.f};
    int i = 1;
    out[i++] = rt_sphere_desc{0.f, 1.f, 0.f, 1.f, RT_MAT_DIELECTRIC, 0.f, 0.f, 0.f, 1.5f};
    out[i++] = rt_sphere_desc{-4.f, 1.f, 0.f, 1.f, RT_MAT_LAMBERTIAN, 0.4f, 0.2f, 0.1f, 0.f};
    out[i++] = rt_sphere_desc{4.f, 1.f, 0.f, 1.f, RT_MAT_METAL, 0.7f, 0.6f, 0.5f, 0.f};
    const int spheres_per_dim = (int)sqrtf((float)n - 4);     // main.cu:160
    const double spacing = 20. / spheres_per_dim;              // main.cu:161
    for (double a = -10; a < 10; a += spacing) {
        for (double b = -10; b < 10 && i < n; b += spacing) {
            const float choose_mat = fp16 ? round_half(RND()) : RND();
            const float th_lambert = fp16 ? round_half(0.8f) : 0.8f, th_metal = fp16 ? round_half(0.95f) : 0.95f;
            rt_sphere_desc s{};
            s.cx = (float)(a + (double)RND());
            s.cy = radius;
            s.cz = (float)(b + (double)RND());
            s.radius = radius;
            if (choose_mat < th_lambert) {
                s.mat = RT_MAT_LAMBERTIAN;
                const float q0 = RND(), q1 = RND(), q2 = RND(), q3 = RND(), q4 = RND(), q5 = RND();
                s.ax = q0 * q1; s.ay = q2 * q3; s.az = q4 * q5;
            } else if (choose_mat < th_metal) {
                s.mat = RT_MAT_METAL;
                const float q0 = RND(), q1 = RND(), q2 = RND(), q3 = RND();
                s.ax = 0.5f * (1.0f + q0); s.ay = 0.5f * (1.0f + q1); s.az = 0.5f * (1.0f + q2);
                const float f = 0.5f * q3;
                s.param = f < 1.0f ? f : 1.0f;                  // material.h:67
            } else {
                s.mat = RT_MAT_DIELECTRIC;
                s.param = 1.5f;
            }
            out[i++] = s;
        }
    }
    if (fp16)
        for (auto &s : out) {
            s.cx = round_half(s.cx); s.cy = round_half(s.cy); s.cz = round_half(s.cz); s.radius = round_half(s.radius);
            s.ax = round_half(s.ax); s.ay = round_half(s.ay); s.az = round_half(s.az); s.param = round_half(s.param);
        }
}

__global__ void k_split_scene(const rt_sphere_desc *__restrict__ d, int n, float4 *__restrict__ geom, float4 *__restrict__ matl, int *__restrict__ tag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const rt_sphere_desc s = d[i];
    geom[i] = make_float4(s.cx, s.cy, s.cz, s.radius);
    matl[i] = make_float4(s.ax, s.ay, s.az, s.param);
    tag[i] = s.mat;
}

// The 36-byte descriptors cross PCIe once, from page-locked staging memory, and are split into the SoA arrays on the device
// (three pageable copies of host-built arrays took 1.0 ms at 100 k spheres: as much as the whole octree build).  The staging
// buffer is also the context's host copy of the scene (rt_scene_download): `src` is copied ONCE, straight into it.
static int upload_scene(rt_context *ctx, const rt_sphere_desc *src, bool clamp_fuzz) {
    const int n = ctx->n;
    CK(ctx->geom.reserve(n));
    CK(ctx->matl.reserve(n));
    CK(ctx->tag.reserve(n));
    const size_t bytes = (size_t)n * sizeof(rt_sphere_desc);
    CK(cudaStreamSynchronize(ctx->stream));                      // (an earlier upload may still be reading the staging buffer)
    CK(ctx->pinned.reserve(bytes, bytes / 4));
    CK(ctx->desc_dev.reserve(bytes, bytes / 4));
    rt_sphere_desc *host = reinterpret_cast<rt_sphere_desc *>(ctx->pinned.ptr);
    memcpy(host, src, bytes);
    if (clamp_fuzz)
        for (int i = 0; i < n; i++)
            if (host[i].mat == RT_MAT_METAL && !(host[i].param < 1.0f)) host[i].param = 1.0f;   // metal::metal clamps fuzz (material.h:67)
    CK(cudaMemcpyAsync(ctx->desc_dev.ptr, ctx->pinned.ptr, bytes, cudaMemcpyHostToDevice, ctx->stream));
    k_split_scene<<<(n + 255) / 256, 256, 0, ctx->stream>>>(reinterpret_cast<const rt_sphere_desc *>(ctx->desc_dev.ptr), n, ctx->geom.ptr,
                                                            ctx->matl.ptr, ctx->tag.ptr);
    CK(cudaGetLastError());
    ctx->octree.built = false;
    return RT_OK;
}

extern "C" int rt_scene_generate(rt_context *ctx, int n, float radius) { return rt_scene_generate_ex(ctx, n, radius, RT_PREC_FP32); }

extern "C" int rt_scene_generate_ex(rt_context *ctx, int n, float radius, int precision) {
    if (!ctx || n < 4) return fail(ctx, RT_ERR_INVALID, "rt_scene_generate: n must be >= 4");
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_scene_generate: unknown precision");
    CK(cudaSetDevice(ctx->device));
    ctx->n = n;
    ctx->half_valid = false;          // the half copy of the scene (USE_FP16 path) is derived on demand
    ctx->list_accel_valid = false;
    std::vector<rt_sphere_desc> world;
    generate_world(n, radius, precision == RT_PREC_FP16, world);
    return upload_scene(ctx, world.data(), false);
}

extern "C" int rt_scene_upload(rt_context *ctx, const rt_sphere_desc *spheres, int n) {
    if (!ctx || !spheres || n < 1) return fail(ctx, RT_ERR_INVALID, "rt_scene_upload: bad arguments");
    CK(cudaSetDevice(ctx->device));
    ctx->n = n;
    ctx->half_valid = false;          // the half copy of the scene (USE_FP16 path) is derived on demand
    ctx->list_accel_valid = false;
    return upload_scene(ctx, spheres, true);
}

extern "C" int rt_scene_download(rt_context *ctx, rt_sphere_desc *out, int n) {
    if (!ctx || !out || n != ctx->n) return fail(ctx, RT_ERR_INVALID, "rt_scene_download: n does not match the scene");
    memcpy(out, ctx->pinned.ptr, (size_t)n * sizeof(rt_sphere_desc));      // the staging buffer of the last upload
    return RT_OK;
}

extern "C" int rt_scene_size(const rt_context *ctx) { return ctx ? ctx->n : 0; }

// ---- camera -----------------------------------------------------------------------------------------------------
// camera.h:22-44 evaluated on the device (same libdevice tanf as the reference).  In the reference every argument
// but the aspect ratio is a compile-time constant, so nvcc folds w, u, v with one rounding per operation; the
// aspect-dependent part keeps the fused form seen in the SASS (DESIGN.md §4).
__global__ void k_camera_setup(rt_camera_desc c, CameraData *out) {
    const float lens_radius = __fdiv_rn(c.aperture, 2.0f);
    const float theta = __fdiv_rn(__fmul_rn(c.vfov, 3.14159265358979323846f), 180.0f);
    const float arg = __fdiv_rn(theta, 2.0f);
    const float half_height = tanf(arg);
    const float half_width = __fmul_rn(c.aspect, half_height);
    float w[3], u[3], v[3];
    {
        const float d[3] = {__fsub_rn(c.lookfrom[0], c.lookat[0]), __fsub_rn(c.lookfrom[1], c.lookat[1]),
                            __fsub_rn(c.lookfrom[2], c.lookat[2])};
        const float l = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(d[0], d[0]), __fmul_rn(d[1], d[1])), __fmul_rn(d[2], d[2])));
        for (int k = 0; k < 3; k++) w[k] = __fdiv_rn(d[k], l);
        // cross(vup, w): vec3.h:95-99
        const float cx = __fsub_rn(__fmul_rn(c.vup[1], w[2]), __fmul_rn(c.vup[2], w[1]));
        const float cy = -__fsub_rn(__fmul_rn(c.vup[0], w[2]), __fmul_rn(c.vup[2], w[0]));
        const float cz = __fsub_rn(__fmul_rn(c.vup[0], w[1]), __fmul_rn(c.vup[1], w[0]));
        const float lc = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz)));
        u[0] = __fdiv_rn(cx, lc); u[1] = __fdiv_rn(cy, lc); u[2] = __fdiv_rn(cz, lc);
        v[0] = __fsub_rn(__fmul_rn(w[1], u[2]), __fmul_rn(w[2], u[1]));
        v[1] = -__fsub_rn(__fmul_rn(w[0], u[2]), __fmul_rn(w[2], u[0]));
        v[2] = __fsub_rn(__fmul_rn(w[0], u[1]), __fmul_rn(w[1], u[0]));
    }
    const float hw = __fmul_rn(half_width, c.focus_dist), hh = __fmul_rn(half_height, c.focus_dist);
    const float h2 = __fmul_rn(__fmul_rn(2.0f, half_width), c.focus_dist);
    const float v2 = __fmul_rn(__fmul_rn(2.0f, half_height), c.focus_dist);
    for (int k = 0; k < 3; k++) {
        out->origin[k] = c.lookfrom[k];
        out->u[k] = u[k]; out->v[k] = v[k]; out->w[k] = w[k];
        float t = __fmaf_rn(-hw, u[k], c.lookfrom[k]);
        t = __fmaf_rn(-hh, v[k], t);
        out->lower_left_corner[k] = __fsub_rn(t, __fmul_rn(c.focus_dist, w[k]));
        out->horizontal[k] = __fmul_rn(h2, u[k]);
        out->vertical[k] = __fmul_rn(v2, v[k]);
    }
    out->lens_radius = lens_radius;
}

extern "C" int rt_camera_set(rt_context *ctx, const rt_camera_desc *desc, int nx, int ny) {
    if (!ctx || nx < 1 || ny < 1) return fail(ctx, RT_ERR_INVALID, "rt_camera_set: bad image size");
    CK(cudaSetDevice(ctx->device));
    rt_camera_desc c;
    if (desc) {
        c = *desc;
    } else {   // main.cu:192-202
        const float lf[3] = {13, 2, 3}, la[3] = {0, 0, 0}, up[3] = {0, 1, 0};
        memcpy(c.lookfrom, lf, sizeof lf); memcpy(c.lookat, la, sizeof la); memcpy(c.vup, up, sizeof up);
        c.vfov = 30.0f;
        c.aspect = (float)nx / (float)ny;
        c.aperture = 0.1f;
        c.focus_dist = 10.0f;
    }
    ctx->cam_desc = c;
    ctx->cam_desc_custom = desc != nullptr;
    ctx->cam_h_nx = ctx->cam_h_ny = 0;          // the half camera is derived on demand
    k_camera_setup<<<1, 1, 0, ctx->stream>>>(c, ctx->cam_dev.ptr);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&ctx->cam_host, ctx->cam_dev.ptr, sizeof(CameraData), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_camera = true;
    ctx->cam_nx = nx; ctx->cam_ny = ny;
    return RT_OK;
}

extern "C" int rt_camera_get(rt_context *ctx, float out22[22]) {
    if (!ctx || !out22 || !ctx->have_camera) return fail(ctx, RT_ERR_STATE, "rt_camera_get: no camera set");
    memcpy(out22, &ctx->cam_host, 22 * sizeof(float));
    return RT_OK;
}

static int ensure_half_camera(rt_context *ctx, int nx, int ny) {
    if (!ctx->have_camera) {
        const int rc = rt_camera_set(ctx, nullptr, nx, ny);
        if (rc) return rc;
    }
    CK(ctx->cam_h.reserve(22));
    if (ctx->cam_h_nx != nx || ctx->cam_h_ny != ny) {
        const rt_camera_desc &c = ctx->cam_desc;
        CK(launch_camera_setup_half(c.lookfrom, c.lookat, c.vup, c.vfov, nx, ny, ctx->cam_desc_custom ? c.aspect : 0.f, c.aperture,
                                    c.focus_dist, ctx->cam_h.ptr, ctx->stream));
        ctx->cam_h_nx = nx; ctx->cam_h_ny = ny;
    }
    return RT_OK;
}

extern "C" int rt_camera_get_half(rt_context *ctx, int nx, int ny, float out22[22]) {
    if (!ctx || !out22 || nx < 1 || ny < 1) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_half: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int rc = ensure_half_camera(ctx, nx, ny);
    if (rc) return rc;
    __half h[22];
    CK(cudaMemcpyAsync(h, ctx->cam_h.ptr, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (int k = 0; k < 22; k++) out22[k] = __half2float(h[k]);
    return RT_OK;
}

// ---- octree -----------------------------------------------------------------------------------------------------
extern "C" int rt_octree_build(rt_context *ctx, int spl, rt_octree_stats *stats) { return rt_octree_build_ex(ctx, spl, RT_PREC_FP32, stats); }

extern "C" int rt_octree_build_ex(rt_context *ctx, int spl, int precision, rt_octree_stats *stats) {
    if (!ctx || spl < 1) return fail(ctx, RT_ERR_INVALID, "rt_octree_build: SPHERES_PER_LEAF must be >= 1");
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_octree_build: unknown precision");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_octree_build: no scene");
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    CK(ctx->octree.build(ctx->stream, ctx->geom.ptr, ctx->tag.ptr, ctx->n, spl, ctx->grid_density, precision == RT_PREC_FP16));
    ctx->half_pairs.valid = false;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        stats->build_ms = ms;
        stats->node_count = ctx->octree.counts.node_count;
        stats->entries = (int64_t)ctx->octree.stats_h[0];
        stats->dropped_full = (int64_t)ctx->octree.stats_h[1];
        stats->dropped_outside = (int64_t)ctx->octree.stats_h[2];
        stats->fine_voxels = ctx->octree.total_voxels;
        stats->fine_refs = ctx->octree.total_refs;
        stats->leaf_count = 0;   // known once the reference layout is exported
    }
    return RT_OK;
}

extern "C" size_t rt_octree_reference_bytes(int spl) { return OctreeBuilder::reference_bytes(spl); }

extern "C" size_t rt_octree_reference_bytes_ex(int spl, int precision) {
    if (spl < 1 || (precision != RT_PREC_FP32 && precision != RT_PREC_FP16)) return 0;
    return OctreeBuilder::reference_bytes(spl, precision == RT_PREC_FP16);
}

extern "C" int rt_octree_export_reference(rt_context *ctx, void *host_blob, size_t bytes) {
    if (!ctx || !host_blob) return RT_ERR_INVALID;
    if (!ctx->octree.built) return fail(ctx, RT_ERR_STATE, "rt_octree_export_reference: build the octree first");
    if (ctx->octree.fp16) {      // the USE_FP16 AABB holds the planes as halves: they must be exact there (k_blob_nodes)
        const float *pl = &ctx->octree.planes.p[0][0];
        for (int k = 0; k < 3 * kPlanes; k++)
            if (__half2float(__float2half_rn(pl[k])) != pl[k])
                return fail(ctx, RT_ERR_UNSUPPORTED, "rt_octree_export_reference: box plane %g is not exact in half", (double)pl[k]);
    }
    CK(cudaSetDevice(ctx->device));
    CK(ctx->octree.export_reference(ctx->stream, host_blob, bytes));
    return RT_OK;
}

extern "C" size_t rt_octree_debug_read(rt_context *ctx, int which, void *host, size_t cap) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    return ctx->octree.debug_read(ctx->stream, which, host, cap);
}

// ---- USE_FP16 state -------------------------------------------------------------------------------------------------
// What the half kernels read, derived on demand and kept until the scene, the tree or the frame size changes: always the scene
// rounded to half; with kHalfPairs the pair lists of one mode (octree: the cells of `tv`; flat: all spheres); with kHalfCamera
// the half camera of an nx x ny frame.  The render and the per-ray entry points share it.
enum { kHalfPairs = 1, kHalfCamera = 2 };
static int ensure_half(rt_context *ctx, unsigned what, bool octree, const TreeView &tv, int nx, int ny) {
    // (a scene change clears half_valid, so the contents a growth drops are never marked valid)
    CK(ctx->geom_h.reserve(ctx->n));
    CK(ctx->matl_h.reserve(ctx->n));
    if (!ctx->half_valid) {
        CK(launch_scene_to_half(ctx->geom.ptr, ctx->matl.ptr, ctx->n, ctx->geom_h.ptr, ctx->matl_h.ptr, ctx->stream));
        ctx->half_valid = true;
        ctx->half_pairs.valid = false;
    }
    if ((what & kHalfPairs) && (!ctx->half_pairs.valid || ctx->half_pairs.octree != octree))
        CK(build_half_pairs(ctx->half_pairs, ctx->geom_h.ptr, ctx->tag.ptr, ctx->n, octree, tv, ctx->stream));
    if (what & kHalfCamera) return ensure_half_camera(ctx, nx, ny);
    return RT_OK;
}

// The structure a render or a per-ray query walks, shared by both so that rt_trace_rays answers a ray as the render's kernels do.
// Octree mode: the octree's grid.  Flat-list mode: hitable_list::hit is "closest over all spheres"; in FP32 from kListGridMinSpheres
// spheres on the grid over ALL spheres answers it with a few dozen tests instead of N (the same minimum; variant 20 forces the N-test
// sweep), built on first use (an undefined slot 0 stays unhittable there too: the build sees its tag, TreeView::slot0_none).
// p.coop_items: four candidates per lane for the cooperative walk once voxel lists are long.
static int select_walk(rt_context *ctx, const bool use_octree, const int precision, const int variant, RenderLaunch &p, bool &list_grid) {
    list_grid = !use_octree && precision == RT_PREC_FP32 && ctx->n >= kListGridMinSpheres && variant != 20;
    if (use_octree) p.tree = ctx->octree.view();
    if (list_grid) {
        if (!ctx->list_accel_valid) {
            CK(ctx->list_accel.build(ctx->stream, ctx->geom.ptr, ctx->tag.ptr, ctx->n, 30, ctx->grid_density, false, true));
            ctx->list_accel_valid = true;
        }
        p.tree = ctx->list_accel.view();
    }
    const OctreeBuilder &acc = list_grid ? ctx->list_accel : ctx->octree;
    p.coop_items = (use_octree || list_grid) && acc.total_voxels > 0 && acc.total_refs / acc.total_voxels >= 40 ? 4 : 2;
    return RT_OK;
}

// ---- render -----------------------------------------------------------------------------------------------------
struct ProgressiveIO {
    uint32_t *state = nullptr;     // 6 words per pixel, device
    bool first = true;
    uint32_t *counts = nullptr;    // with a pixel list (rt_render_pixels_progressive): samples per frame pixel, or nullptr
};
struct PixelList {                 // rt_render_pixels: render these pixels of the frame, results in list order
    const uint32_t *pixels = nullptr;      // device
    int count = 0;
};
// device (or managed) memory of the context's GPU: a kernel may dereference it
static bool on_device(const rt_context *ctx, const void *ptr) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged) && at.device == ctx->device;
}
// Statistics of the context's last render: its counters, kernel, launch count and the device time between its events.  Waits
// for the context's stream.
static int read_render_stats(rt_context *ctx, rt_render_stats *stats) {
    unsigned long long c[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(c, ctx->counters.ptr, sizeof c, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memset(stats, 0, sizeof *stats);
    stats->rays = c[0]; stats->paths = c[1];
    stats->sphere_tests = c[2]; stats->node_tests = c[3];   // zero unless built with -DRT_COUNTERS
    stats->kernel_id = ctx->last_kernel;
    stats->launches = ctx->last_launches;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) stats->kernel_ms = ms;
    return RT_OK;
}
static int do_render(rt_context *ctx, const rt_render_args *a, float *out_dev, bool finalize, rt_render_stats *stats,
                     const ProgressiveIO *prog = nullptr, const PixelList *list = nullptr) {
    if (!ctx || !a || !out_dev) return fail(ctx, RT_ERR_INVALID, "render: null argument");
    if (a->nx < 1 || a->ny < 1 || a->ns < 1) return fail(ctx, RT_ERR_INVALID, "render: bad nx/ny/ns");
    // a pixel list with progressive state: rt_render_pixels_progressive (frame-indexed sums, states and counts)
    const bool list_prog = list && prog;
    if (list) {
        if (!list->pixels || list->count < 1) return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: null pixel list or count < 1");
        if (a->shard_mode != RT_SHARD_NONE) return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: pixel lists are not sharded (give each GPU its own list)");
        if (!on_device(ctx, list->pixels) || !on_device(ctx, out_dev))
            return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: pixels_dev and out_dev must be device memory of the context's GPU");
        if (list_prog && (!on_device(ctx, prog->state) || (prog->counts && !on_device(ctx, prog->counts))))
            return fail(ctx, RT_ERR_INVALID, "rt_render_pixels_progressive: rng_state_dev and counts_dev must be device memory of the context's GPU");
    }
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "render: no scene (rt_scene_generate / rt_scene_upload first)");
    if (a->use_octree && !ctx->octree.built) return fail(ctx, RT_ERR_STATE, "render: USE_OCTREE set but no octree built");
    if (a->seed_mode != RT_SEED_HEAD && a->seed_mode != RT_SEED_UPSTREAM) return fail(ctx, RT_ERR_INVALID, "render: unknown seed_mode");
    if (a->precision != RT_PREC_FP32 && a->precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "render: unknown precision");
    const bool fp16 = a->precision == RT_PREC_FP16;
    // a tile shard holds whole pixels' half sums, exact in float, so shards add up to the 1-GPU frame; the half sum of ns/G
    // samples per rank is a different image from any build of the reference
    if (fp16 && a->shard_mode == RT_SHARD_SPP)
        return fail(ctx, RT_ERR_UNSUPPORTED, "render: USE_FP16 frames shard by tiles only (RT_SHARD_TILES): spp shards' half sums do not add up to the 1-GPU frame");
    if (a->use_octree && ctx->octree.built && ctx->octree.fp16 != fp16)
        return fail(ctx, RT_ERR_STATE, "render: the octree was built for the other precision (rt_octree_build_ex)");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->have_camera || ctx->cam_nx != a->nx || ctx->cam_ny != a->ny) {
        // only the default main.cu camera follows the frame size (its aspect ratio is nx/ny, main.cu:198); a description
        // given through rt_camera_set(desc) / rt_apply_camera is kept as it is, aspect included
        const rt_camera_desc keep = ctx->cam_desc;
        const int rc = rt_camera_set(ctx, ctx->have_camera && ctx->cam_desc_custom ? &keep : nullptr, a->nx, a->ny);
        if (rc) return rc;
    }
    const int count = a->shard_mode == RT_SHARD_NONE ? 1 : (a->shard_count < 1 ? 1 : a->shard_count);
    const int rank = a->shard_mode == RT_SHARD_NONE ? 0 : a->shard_rank;
    if (rank < 0 || rank >= count) return fail(ctx, RT_ERR_INVALID, "render: shard_rank out of range");
    if (finalize && count > 1) return fail(ctx, RT_ERR_INVALID, "render: a sharded frame must go through rt_render_accumulate");

    RenderLaunch p;
    memset(&p, 0, sizeof p);
    p.scene.geom = ctx->geom.ptr; p.scene.matl = ctx->matl.ptr; p.scene.tag = ctx->tag.ptr; p.scene.n = ctx->n;
    bool list_grid = false;
    {
        const int rc = select_walk(ctx, a->use_octree != 0, a->precision, a->tune[1], p, list_grid);
        if (rc) return rc;
    }
    p.cam = ctx->cam_host;                        // per-context camera, by value in the launch parameters
    p.nx = a->nx; p.ny = a->ny;
    p.ns_total = a->ns;
    p.ns_local = a->ns;
    p.max_depth = a->max_depth > 0 ? a->max_depth : 50;
    p.tiles_x = (a->nx + 7) / 8;
    const long long tiles_y = (a->ny + 3) / 4;
    const long long ntiles = (long long)p.tiles_x * tiles_y;
    p.tile_first = 0; p.tile_stride = 1;
    long long owned = ntiles;
    const size_t fb_bytes = (size_t)a->nx * a->ny * 3 * sizeof(float);
    const bool continuing = prog && !prog->first;
    if (a->shard_mode == RT_SHARD_TILES && count > 1) {
        p.tile_first = rank; p.tile_stride = count;
        owned = (ntiles - rank + count - 1) / count;
        if (!continuing) CK(cudaMemsetAsync(out_dev, 0, fb_bytes, ctx->stream));       // pixels of other shards stay 0 so shards add up
    } else if (a->shard_mode == RT_SHARD_SPP && count > 1) {
        p.ns_local = a->ns / count + (rank < a->ns % count ? 1 : 0);
        // shard g draws from streams seeded 1984 + pixel_index + g*num_pixels: distinct seeds, the reference's own
        // convention for independent streams (main.cu:91-93); g = 0 is the reference stream
        p.seed_offset = (unsigned long long)rank * (unsigned long long)a->nx * (unsigned long long)a->ny;
        if (p.ns_local == 0) {
            if (!continuing) CK(cudaMemsetAsync(out_dev, 0, fb_bytes, ctx->stream));
            if (stats) memset(stats, 0, sizeof *stats);
            return RT_OK;
        }
    }
    if (owned * 32 > 0xfffffff0ll) return fail(ctx, RT_ERR_INVALID, "render: image too large for the 32-bit work queue");
    const size_t npix = (size_t)a->nx * a->ny;
    if (list_prog) {        // scratch for the preparation pass, before anything is launched
        CK(ctx->list_dedup.reserve((size_t)list->count));
        CK(ctx->list_mask.reserve((npix + 31) / 32));
    }
    p.total_items = list ? (uint32_t)list->count : (uint32_t)(owned * 32);
    if (list) p.pixels = list_prog ? ctx->list_dedup.ptr : list->pixels;
    p.finalize = finalize ? 1 : 0;
    p.variant = a->tune[1] ? a->tune[1] : ctx->default_variant;
    p.out = out_dev;
    p.work_counter = ctx->work_counter.ptr;
    p.counters = ctx->counters.ptr;
    CK(cudaMemsetAsync(ctx->counters.ptr, 0, 32 * 8, ctx->stream));
    int blocks = 0;
    int launches = 1;
    const int mode = list_prog ? kModeListProgressive : list ? kModeList : kModeFrame;
    if (a->seed_mode == RT_SEED_UPSTREAM && !continuing) {
        if (!ctx->skip_tables.ptr) {
            const std::vector<uint32_t> &t = host_skip_tables();
            CK(ctx->skip_tables.reserve(t.size()));
            CK(cudaMemcpyAsync(ctx->skip_tables.ptr, t.data(), t.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        }
        if (!list_prog) {       // (a progressive list seeds its pixels straight into the caller's state buffer)
            const size_t nstates = list ? (size_t)list->count : npix;      // stream states to seed
            CK(ctx->seed_states.reserve(nstates * 6));
            p.seed_states = ctx->seed_states.ptr;
        }
    }
    if (list_prog) {
        p.seed_states = prog->state;                  // read and stored back by the list-progressive instances
        p.accumulate = continuing ? 1 : 0;
    } else if (prog) {
        p.state_out = prog->state;
        p.accumulate = continuing ? 1 : 0;
    }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (list_prog) {
        launches = 2;       // the preparation pass, launched right before the render (below)
    } else if (continuing) {
        p.seed_states = prog->state;                  // every pixel resumes its own stream
    } else if (p.seed_states) {   // render_init (main.cu:424): inside the timed region, as in the reference
        if (list)                 // only the listed pixels' streams
            CK(launch_seed_upstream_list(ctx->seed_states.ptr, list->pixels, list->count, (size_t)a->nx * a->ny, 1984ull, ctx->skip_tables.ptr,
                                         ctx->stream));
        else                      // spp shard g draws from subsequences pixel_index + g * num_pixels (g = 0: the reference's streams)
            CK(launch_seed_upstream(ctx->seed_states.ptr, (size_t)a->nx * a->ny, 1984ull, p.seed_offset, ctx->skip_tables.ptr, ctx->stream));
        launches = 2;
    }
    if (fp16) {
        {
            const int rc = ensure_half(ctx, kHalfPairs | kHalfCamera, a->use_octree != 0, p.tree, a->nx, a->ny);
            if (rc) return rc;
        }
    }
    // rt_render_pixels_progressive: dedupe, counts and (first) seeding, inside the timed region as the frames' seeding, and after
    // the last step that can fail on the context's side, so that an error leaves the caller's buffers untouched
    if (list_prog)
        CK(launch_pixels_progressive_prep(list->pixels, list->count, (uint32_t)npix, ctx->list_mask.ptr, ctx->list_dedup.ptr, prog->counts,
                                          (uint32_t)a->ns, prog->first, prog->state, a->seed_mode == RT_SEED_UPSTREAM ? ctx->skip_tables.ptr : nullptr,
                                          ctx->stream));
    if (fp16) {
        CK(launch_render_half(p, a->use_octree != 0, ctx->geom_h.ptr, ctx->matl_h.ptr, ctx->cam_h.ptr, ctx->half_pairs, ctx->prop.multiProcessorCount,
                              ctx->stream, &blocks, mode));
        ctx->last_kernel = kKernelHalf;
    } else {
        CK(launch_render(p, a->use_octree != 0 || list_grid, ctx->prop.multiProcessorCount, ctx->prop.sharedMemPerBlockOptin, ctx->stream, &blocks,
                         &ctx->last_kernel, mode));
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    ctx->last_launches = launches;
    return stats ? read_render_stats(ctx, stats) : RT_OK;
}

// curand_init(seed, subsequence, 0) -> {d, v0..v4}: host-side evaluation with the library's own skip matrices (no GPU needed)
extern "C" int rt_xorwow_state(unsigned long long seed, unsigned long long subsequence, uint32_t out6[6]) {
    if (!out6 || (subsequence >> kSkipBits)) return RT_ERR_INVALID;
    xorwow s;
    xorwow_seed_subsequence(s, seed, subsequence, host_skip_tables().data());
    out6[0] = s.d; out6[1] = s.v0; out6[2] = s.v1; out6[3] = s.v2; out6[4] = s.v3; out6[5] = s.v4;
    return RT_OK;
}

// Statistics of the LAST render call, for callers that passed stats = NULL to keep the call asynchronous (e.g. to queue the
// multi-GPU exchange behind the render without a host round trip in between): waits for the context's stream, then reads the
// counters and the render's CUDA events.
extern "C" int rt_last_render_stats(rt_context *ctx, rt_render_stats *stats) {
    if (!ctx || !stats) return fail(ctx, RT_ERR_INVALID, "rt_last_render_stats: null argument");
    CK(cudaSetDevice(ctx->device));
    return read_render_stats(ctx, stats);
}

// test hook: the raw device counters of the last render
extern "C" int rt_debug_counters(rt_context *ctx, uint64_t out[32]) {
    if (!ctx || !out) return fail(ctx, RT_ERR_INVALID, "rt_debug_counters: null argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->counters.ptr, 32 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// One host array of a per-ray query.  `in`: copied to the device before the launch; `out`: copied back after it (zero-filled
// before, so what the kernel leaves unwritten comes back as zeros); both: copied in and back (the XORWOW states).
struct HostArray {
    const void *in;
    void *out;
    size_t bytes;
};
template <typename T> static HostArray stage_in(const T *h, size_t count) { return HostArray{h, nullptr, count * sizeof(T)}; }
template <typename T> static HostArray stage_out(T *h, size_t count) { return HostArray{nullptr, h, count * sizeof(T)}; }
template <typename T> static HostArray stage_inout(T *h, size_t count) { return HostArray{h, h, count * sizeof(T)}; }
struct DevPtr {                    // a staged array's device address, handed to a launcher as the pointer type it takes
    void *p;
    template <typename T> operator T *() const { return static_cast<T *>(p); }
};

// Runs one per-ray query on the context's stream: stages `arrays` in one device allocation (each at a 16-byte aligned offset:
// the states are read as uint2), calls launch(dev) with their device addresses in the order given, copies the results back and
// synchronises once.  The allocation is released on every exit path.
template <typename Launch>
static int run_staged(rt_context *ctx, std::initializer_list<HostArray> arrays, Launch launch) {
    auto padded = [](size_t bytes) { return (bytes + 15) & ~(size_t)15; };
    size_t total = 0;
    for (const HostArray &a : arrays) total += padded(a.bytes);
    Buffer<char> buf;
    CK(buf.reserve(total));
    char *base = buf.ptr;
    std::vector<DevPtr> dev;
    size_t off = 0;
    for (const HostArray &a : arrays) {
        if (a.in) CK(cudaMemcpyAsync(base + off, a.in, a.bytes, cudaMemcpyHostToDevice, ctx->stream));
        else CK(cudaMemsetAsync(base + off, 0, a.bytes, ctx->stream));
        dev.push_back(DevPtr{base + off});
        off += padded(a.bytes);
    }
    CK(launch(dev.data()));
    off = 0;
    for (const HostArray &a : arrays) {
        if (a.out) CK(cudaMemcpyAsync(a.out, base + off, a.bytes, cudaMemcpyDeviceToHost, ctx->stream));
        off += padded(a.bytes);
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// test hook: closest hit of caller-supplied rays (host arrays of 3 floats per ray), by the walk the render would use for the scene
// (select_walk; RT_RENDER_VARIANT picks another: launch_trace_rays)
extern "C" int rt_trace_rays(rt_context *ctx, int use_octree, int n, const float *org, const float *dir, int *out_idx, float *out_t) {
    return rt_trace_rays_ex(ctx, use_octree, RT_PREC_FP32, n, org, dir, out_idx, out_t);
}

// camera::get_ray (camera.h:45-49) for n (s, t) pairs: each draws its lens sample from ITS OWN XORWOW state (6 words, in/out)
extern "C" int rt_camera_get_rays(rt_context *ctx, int n, const float *s, const float *t, uint32_t *states6, float *org, float *dir) {
    return rt_camera_get_rays_ex(ctx, RT_PREC_FP32, n, s, t, states6, org, dir);
}

// material::scatter (material.h:55-113) + the hit record of sphere::hit (sphere.h:30-33) for n (ray, sphere, t) triples
extern "C" int rt_scatter_rays(rt_context *ctx, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                               uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten, int *scattered) {
    return rt_scatter_rays_ex(ctx, RT_PREC_FP32, n, sphere_idx, org, dir, t_hit, states6, out_p, out_normal, out_dir, out_atten, scattered);
}

// ---- the same three queries under a given arithmetic ----------------------------------------------------------------------
// RT_PREC_FP16: the USE_FP16 build's hitTree / hitable_list::hit, camera::get_ray and material::scatter (rt_render_half.cuh):
// float inputs are rounded to half on entry, outputs are halves widened to float.
extern "C" int rt_trace_rays_ex(rt_context *ctx, int use_octree, int precision, int n, const float *org, const float *dir, int *out_idx,
                                float *out_t) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays_ex: unknown precision");
    if (!ctx || n < 1 || !org || !dir || !out_idx || !out_t) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays_ex: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: no scene");
    if (use_octree && !ctx->octree.built) return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: no octree built");
    const bool fp16 = precision == RT_PREC_FP16;
    if (use_octree && ctx->octree.fp16 != fp16)
        return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: the octree was built for the other precision (rt_octree_build_ex)");
    CK(cudaSetDevice(ctx->device));
    RenderLaunch p;
    memset(&p, 0, sizeof p);
    p.scene.geom = ctx->geom.ptr; p.scene.matl = ctx->matl.ptr; p.scene.tag = ctx->tag.ptr; p.scene.n = ctx->n;
    p.variant = fp16 ? 0 : ctx->default_variant;     // RT_RENDER_VARIANT selects the FP32 walk (launch_trace_rays)
    bool list_grid = false;
    {
        const int rc = select_walk(ctx, use_octree != 0, precision, p.variant, p, list_grid);
        if (rc) return rc;
    }
    if (fp16) {
        const int rc = ensure_half(ctx, kHalfPairs, use_octree != 0, p.tree, 0, 0);
        if (rc) return rc;
    }
    const size_t N = (size_t)n;
    return run_staged(ctx, {stage_in(org, 3 * N), stage_in(dir, 3 * N), stage_out(out_idx, N), stage_out(out_t, N)}, [&](const DevPtr *d) {
        return fp16 ? launch_trace_rays_half(p, use_octree != 0, ctx->geom_h.ptr, ctx->half_pairs, d[0], d[1], n, d[2], d[3], ctx->stream)
                    : launch_trace_rays(p, use_octree != 0 || list_grid, d[0], d[1], n, d[2], d[3], ctx->stream);
    });
}

extern "C" int rt_camera_get_rays_ex(rt_context *ctx, int precision, int n, const float *s, const float *t, uint32_t *states6, float *org,
                                     float *dir) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_rays_ex: unknown precision");
    if (!ctx || n < 1 || !s || !t || !states6 || !org || !dir) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_rays_ex: bad arguments");
    if (!ctx->have_camera) return fail(ctx, RT_ERR_STATE, "rt_camera_get_rays_ex: no camera set (rt_camera_set)");
    CK(cudaSetDevice(ctx->device));
    const bool fp16 = precision == RT_PREC_FP16;
    if (fp16) {
        const int rc = ensure_half_camera(ctx, ctx->cam_nx, ctx->cam_ny);      // the camera the FP16 render of this frame size uses
        if (rc) return rc;
    }
    const size_t N = (size_t)n;
    return run_staged(ctx, {stage_in(s, N), stage_in(t, N), stage_inout(states6, 6 * N), stage_out(org, 3 * N), stage_out(dir, 3 * N)},
                      [&](const DevPtr *d) {
                          return fp16 ? launch_camera_rays_half(ctx->cam_h.ptr, n, d[0], d[1], d[2], d[3], d[4], ctx->stream)
                                      : launch_camera_rays(ctx->cam_host, n, d[0], d[1], d[2], d[3], d[4], ctx->stream);
                      });
}

extern "C" int rt_scatter_rays_ex(rt_context *ctx, int precision, int n, const int *sphere_idx, const float *org, const float *dir,
                                  const float *t_hit, uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten,
                                  int *scattered) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_scatter_rays_ex: unknown precision");
    if (!ctx || n < 1 || !sphere_idx || !org || !dir || !t_hit || !states6 || !out_p || !out_normal || !out_dir || !out_atten || !scattered)
        return fail(ctx, RT_ERR_INVALID, "rt_scatter_rays_ex: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_scatter_rays_ex: no scene");
    CK(cudaSetDevice(ctx->device));
    const bool fp16 = precision == RT_PREC_FP16;
    if (fp16) {
        const TreeView none{};
        const int rc = ensure_half(ctx, 0u, false, none, 0, 0);
        if (rc) return rc;
    }
    SceneView sv;
    sv.geom = ctx->geom.ptr; sv.matl = ctx->matl.ptr; sv.tag = ctx->tag.ptr; sv.n = ctx->n;
    const size_t N = (size_t)n;
    return run_staged(ctx, {stage_in(sphere_idx, N), stage_in(org, 3 * N), stage_in(dir, 3 * N), stage_in(t_hit, N), stage_inout(states6, 6 * N),
                            stage_out(out_p, 3 * N), stage_out(out_normal, 3 * N), stage_out(out_dir, 3 * N), stage_out(out_atten, 3 * N),
                            stage_out(scattered, N)},
                      [&](const DevPtr *d) {
                          return fp16 ? launch_scatter_rays_half(sv, ctx->geom_h.ptr, ctx->matl_h.ptr, n, d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7],
                                                                 d[8], d[9], ctx->stream)
                                      : launch_scatter_rays(sv, n, d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7], d[8], d[9], ctx->stream);
                      });
}

extern "C" int rt_render_accumulate(rt_context *ctx, const rt_render_args *args, float *accum_dev, rt_render_stats *stats) {
    return do_render(ctx, args, accum_dev, false, stats);
}

extern "C" int rt_render(rt_context *ctx, const rt_render_args *args, float *fb_dev, rt_render_stats *stats) {
    return do_render(ctx, args, fb_dev, true, stats);
}

extern "C" int rt_render_pixels(rt_context *ctx, const rt_render_args *args, const uint32_t *pixels_dev, int count, float *out_dev,
                                int finalize, rt_render_stats *stats) {
    PixelList list;
    list.pixels = pixels_dev;
    list.count = count;
    return do_render(ctx, args, out_dev, finalize != 0, stats, nullptr, &list);
}

extern "C" int rt_render_pixels_progressive(rt_context *ctx, const rt_render_args *args, const uint32_t *pixels_dev, int count,
                                            float *accum_dev, uint32_t *rng_state_dev, uint32_t *counts_dev, int first, rt_render_stats *stats) {
    if (!rng_state_dev) return fail(ctx, RT_ERR_INVALID, "rt_render_pixels_progressive: null state buffer");
    PixelList list;
    list.pixels = pixels_dev;
    list.count = count;
    ProgressiveIO io;
    io.state = rng_state_dev;
    io.first = first != 0;
    io.counts = counts_dev;
    return do_render(ctx, args, accum_dev, false, stats, &io, &list);
}

extern "C" int rt_render_progressive(rt_context *ctx, const rt_render_args *args, float *accum_dev, uint32_t *rng_state_dev, int first,
                                     rt_render_stats *stats) {
    if (!rng_state_dev) return fail(ctx, RT_ERR_INVALID, "rt_render_progressive: null state buffer");
    ProgressiveIO io;
    io.state = rng_state_dev;
    io.first = first != 0;
    return do_render(ctx, args, accum_dev, false, stats, &io);
}

extern "C" int rt_finalize(rt_context *ctx, const float *accum_dev, float *fb_dev, int nx, int ny, int ns) {
    if (nx < 1 || ny < 1) return fail(ctx, RT_ERR_INVALID, "rt_finalize: bad arguments");
    return rt_finalize_ex(ctx, accum_dev, fb_dev, (size_t)nx * ny * 3, ns, RT_PREC_FP32);
}

extern "C" int rt_finalize_n(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns) {
    return rt_finalize_ex(ctx, accum_dev, fb_dev, count, ns, RT_PREC_FP32);
}

extern "C" int rt_finalize_ex(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns, int precision) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_finalize_ex: unknown precision");
    if (!ctx || !accum_dev || !fb_dev || ns < 1) return fail(ctx, RT_ERR_INVALID, "rt_finalize_ex: bad arguments");
    if (count == 0) return RT_OK;
    CK(cudaSetDevice(ctx->device));
    CK(precision == RT_PREC_FP16 ? launch_finalize_half(accum_dev, fb_dev, count, ns, ctx->stream)
                                 : launch_finalize_n(accum_dev, fb_dev, count, ns, ctx->stream));
    return RT_OK;
}

extern "C" int rt_finalize_counts(rt_context *ctx, const float *accum_dev, const uint32_t *counts_dev, float *fb_dev, size_t npix, int precision) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_finalize_counts: unknown precision");
    if (!ctx || !accum_dev || !counts_dev || !fb_dev) return fail(ctx, RT_ERR_INVALID, "rt_finalize_counts: null argument");
    if (npix == 0) return RT_OK;
    CK(cudaSetDevice(ctx->device));
    if (!on_device(ctx, accum_dev) || !on_device(ctx, counts_dev) || !on_device(ctx, fb_dev))
        return fail(ctx, RT_ERR_INVALID, "rt_finalize_counts: accum_dev, counts_dev and fb_dev must be device memory of the context's GPU");
    CK(launch_finalize_counts(accum_dev, counts_dev, fb_dev, npix, precision == RT_PREC_FP16, ctx->stream));
    return RT_OK;
}

// Adaptive sampling over the frame queue's 8x4 tiles (rt_adaptive.h, rt_adaptive.cu).  Every round lists whole tiles that all
// have the same count, so it is one list-progressive render with one ns; the render kernels and their bit-identity guarantee are
// those of rt_render_progressive and rt_render_pixels_progressive.
extern "C" int rt_render_adaptive(rt_context *ctx, const rt_render_args *args, const rt_adaptive_params *params, float *accum_dev,
                                  uint32_t *rng_state_dev, uint32_t *counts_dev, float *fb_dev, float *err_dev, rt_adaptive_stats *stats) {
    if (!ctx || !args || !params || !accum_dev || !rng_state_dev || !counts_dev || !fb_dev)
        return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: null argument");
    const int min_spp = params->min_spp, max_spp = args->ns;
    const float threshold = params->threshold;
    if (args->nx < 1 || args->ny < 1) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: bad nx/ny");
    if (min_spp < 2 || (min_spp & 1)) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: min_spp must be even and >= 2");
    if (max_spp < min_spp || max_spp > 65536) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: args->ns (max_spp) must be in [min_spp, 65536]");
    if (!(threshold >= 0.0f)) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: threshold must be >= 0 (and not NaN)");
    if (args->shard_mode != RT_SHARD_NONE) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: adaptive frames are not sharded");
    if (args->seed_mode != RT_SEED_HEAD && args->seed_mode != RT_SEED_UPSTREAM) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: unknown seed_mode");
    if (args->precision != RT_PREC_FP32 && args->precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: unknown precision");
    const size_t npix = (size_t)args->nx * args->ny;
    const uint32_t tiles_x = (uint32_t)(args->nx + 7) / 8;
    const unsigned long long tiles = (unsigned long long)tiles_x * (unsigned long long)((args->ny + 3) / 4);
    if (tiles * 32 > 0xfffffff0ull) return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: image too large for the 32-bit work queue");
    if (!on_device(ctx, accum_dev) || !on_device(ctx, rng_state_dev) || !on_device(ctx, counts_dev) || !on_device(ctx, fb_dev) ||
        (err_dev && !on_device(ctx, err_dev)))
        return fail(ctx, RT_ERR_INVALID, "rt_render_adaptive: accum, state, counts, fb and err must be device memory of the context's GPU");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_render_adaptive: no scene (rt_scene_generate / rt_scene_upload first)");
    if (args->use_octree && !ctx->octree.built) return fail(ctx, RT_ERR_STATE, "rt_render_adaptive: USE_OCTREE set but no octree built");
    const bool fp16 = args->precision == RT_PREC_FP16;
    if (args->use_octree && ctx->octree.fp16 != fp16)
        return fail(ctx, RT_ERR_STATE, "rt_render_adaptive: the octree was built for the other precision (rt_octree_build_ex)");
    CK(cudaSetDevice(ctx->device));
    // scratch, before anything is launched: the snapshot, the tile words, the list, the scan's storage, and the rounds' list scratch
    size_t scan_bytes = 0;
    CK(adaptive_scan_temp_bytes((uint32_t)tiles, &scan_bytes));
    CK(ctx->ad_snap.reserve(npix * 3));
    CK(ctx->ad_tiles.reserve((size_t)tiles * 3));
    CK(ctx->ad_list.reserve(npix));
    CK(ctx->ad_scan.reserve(scan_bytes / 4 + 1));
    CK(ctx->list_dedup.reserve(npix));
    CK(ctx->list_mask.reserve((npix + 31) / 32));

    int rc;
    rt_render_stats sum, one;
    memset(&sum, 0, sizeof sum);
    auto render = [&](rt_render_args &ra, const ProgressiveIO &io, const PixelList *list) {
        const int r = do_render(ctx, &ra, accum_dev, false, &one, &io, list);
        sum.rays += one.rays; sum.paths += one.paths; sum.sphere_tests += one.sphere_tests; sum.node_tests += one.node_tests;
        sum.launches += one.launches; sum.kernel_id = one.kernel_id;
        return r;
    };
    CK(cudaEventRecord(ctx->ad_ev0, ctx->stream));
    // two whole-frame segments of min_spp/2 samples, the snapshot between them: the first estimate of every pixel
    rt_render_args ra = *args;
    ra.ns = min_spp / 2;
    ProgressiveIO io;
    io.state = rng_state_dev;
    io.first = true;
    if ((rc = render(ra, io, nullptr))) return rc;
    CK(cudaMemcpyAsync(ctx->ad_snap.ptr, accum_dev, npix * 3 * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    io.first = false;
    if ((rc = render(ra, io, nullptr))) return rc;
    CK(launch_fill_counts(counts_dev, npix, (uint32_t)min_spp, ctx->stream));
    AdaptiveTiles t;
    t.listed = ctx->ad_tiles.ptr; t.offset = ctx->ad_tiles.ptr + tiles; t.done = ctx->ad_tiles.ptr + 2 * tiles;
    t.scan_temp = ctx->ad_scan.ptr; t.scan_temp_bytes = ctx->ad_scan.cap * 4;
    CK(cudaMemsetAsync(t.done, 0, (size_t)tiles * 4, ctx->stream));
    // rounds: the tiles not done all have snapshot count a and count c; a refined tile doubles its count, capped at max_spp, so
    // there are at most ceil(log2(max_spp / min_spp)) <= 15 rounds
    io.counts = counts_dev;
    PixelList list;
    list.pixels = ctx->ad_list.ptr;
    uint32_t a = (uint32_t)min_spp / 2, c = (uint32_t)min_spp;
    int rounds = 0;
    uint64_t round_pixels[16] = {};
    for (;;) {
        uint32_t listed = 0;
        CK(launch_adaptive_select(accum_dev, ctx->ad_snap.ptr, err_dev, args->nx, args->ny, a, c, c < (uint32_t)max_spp, threshold, t,
                                  ctx->ad_list.ptr, &listed, ctx->stream));
        if (listed == 0) break;
        const uint32_t more = c < (uint32_t)max_spp - c ? c : (uint32_t)max_spp - c;
        ra.ns = (int)more;
        list.count = (int)listed;
        if ((rc = render(ra, io, &list))) return rc;
        round_pixels[rounds++] = listed;
        a = c;
        c += more;
    }
    CK(launch_finalize_counts(accum_dev, counts_dev, fb_dev, npix, fp16, ctx->stream));
    CK(cudaEventRecord(ctx->ad_ev1, ctx->stream));
    if (stats) {
        CK(cudaEventSynchronize(ctx->ad_ev1));
        memset(stats, 0, sizeof *stats);
        stats->render = sum;
        float ms = 0;
        if (cudaEventElapsedTime(&ms, ctx->ad_ev0, ctx->ad_ev1) == cudaSuccess) stats->render.kernel_ms = ms;
        stats->rounds = rounds;
        memcpy(stats->round_pixels, round_pixels, sizeof round_pixels);
    }
    return RT_OK;
}

// rt_render into the context's scratch frame, grown to the frame's size: the device frame of the host and PPM outputs
static int render_to_scratch(rt_context *ctx, const rt_render_args *args, rt_render_stats *stats) {
    CK(cudaSetDevice(ctx->device));
    CK(ctx->scratch_fb.reserve((size_t)args->nx * args->ny * 3));
    return do_render(ctx, args, ctx->scratch_fb.ptr, true, stats);
}

extern "C" int rt_render_to_host(rt_context *ctx, const rt_render_args *args, float *fb_host, rt_render_stats *stats) {
    if (!ctx || !args || !fb_host) return fail(ctx, RT_ERR_INVALID, "rt_render_to_host: null argument");
    const int rc = render_to_scratch(ctx, args, stats);
    if (rc) return rc;
    CK(cudaMemcpyAsync(fb_host, ctx->scratch_fb.ptr, (size_t)args->nx * args->ny * 3 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// ---- output on the device (rt_ppm.cu) ---------------------------------------------------------------------------------
extern "C" int rt_ppm_format(rt_context *ctx, const float *fb_dev, int nx, int ny, size_t *len_out) {
    if (!ctx || !fb_dev || nx < 0 || ny < 0) return fail(ctx, RT_ERR_INVALID, "rt_ppm_format: bad argument");
    CK(cudaSetDevice(ctx->device));
    CK(ppm_format_device(ctx->ppm, fb_dev, nx, ny, ctx->stream, len_out));
    return RT_OK;
}

extern "C" int rt_ppm_read(rt_context *ctx, char *buf_host, size_t cap) {
    if (!ctx || !buf_host) return fail(ctx, RT_ERR_INVALID, "rt_ppm_read: null argument");
    if (!ctx->ppm.text.ptr || cap < ctx->ppm.text_len) return fail(ctx, RT_ERR_INVALID, "rt_ppm_read: no formatted frame, or the buffer is smaller than its text");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(buf_host, ctx->ppm.text.ptr, ctx->ppm.text_len, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

extern "C" int rt_render_to_ppm(rt_context *ctx, const rt_render_args *args, rt_render_stats *stats, size_t *len_out) {
    if (!ctx || !args) return fail(ctx, RT_ERR_INVALID, "rt_render_to_ppm: null argument");
    const int rc = render_to_scratch(ctx, args, stats);
    if (rc) return rc;
    CK(ppm_format_device(ctx->ppm, ctx->scratch_fb.ptr, args->nx, args->ny, ctx->stream, len_out));
    return RT_OK;
}

// ---- output: main.cu:321-333 -------------------------------------------------------------------------------------
static inline char *put_int(char *p, int v) {   // what `ostream << int` prints
    char tmp[16];
    int n = 0;
    unsigned u = v < 0 ? 0u - (unsigned)v : (unsigned)v;
    do { tmp[n++] = (char)('0' + u % 10); u /= 10; } while (u);
    if (v < 0) *p++ = '-';
    while (n) *p++ = tmp[--n];
    return p;
}
extern "C" size_t rt_format_ppm(const float *fb, int nx, int ny, char *buf, size_t cap) {
    char head[64];
    const int hl = snprintf(head, sizeof head, "P3\n%d %d\n255\n", nx, ny);
    size_t off = (size_t)hl;
    if (buf && off <= cap) memcpy(buf, head, (size_t)hl);
    char line[48];
    for (int j = ny - 1; j >= 0; j--) {
        for (int i = 0; i < nx; i++) {
            const size_t pi = ((size_t)j * nx + i) * 3;
            char *p = line;
            p = put_int(p, (int)(255.99 * fb[pi + 0])); *p++ = ' ';
            p = put_int(p, (int)(255.99 * fb[pi + 1])); *p++ = ' ';
            p = put_int(p, (int)(255.99 * fb[pi + 2])); *p++ = '\n';
            const size_t len = (size_t)(p - line);
            if (buf && off + len <= cap) memcpy(buf + off, line, len);
            off += len;
        }
    }
    return off;
}

// ---- FP32 roofline denominator: dense FFMA issue rate of this GPU, measured -------------------------------------
__global__ void __launch_bounds__(256) k_ffma_peak(float *out, int iters, float a, float b) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            x0 = __fmaf_rn(x0, a, b); x1 = __fmaf_rn(x1, a, b); x2 = __fmaf_rn(x2, a, b); x3 = __fmaf_rn(x3, a, b);
            x4 = __fmaf_rn(x4, a, b); x5 = __fmaf_rn(x5, a, b); x6 = __fmaf_rn(x6, a, b); x7 = __fmaf_rn(x7, a, b);
        }
    }
    const float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678f) out[0] = s;   // keeps the chain alive, never true in practice
}

// Rate of a peak probe kernel, launch(blocks, threads, iters): its best device time over three runs after a warm-up run, as
// TFLOP/s for `iter_flops` per thread and iteration
template <typename Launch>
static int peak_rate(rt_context *ctx, double iter_flops, float *tflops, float *ms_out, Launch launch) {
    if (!ctx || !tflops) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        launch(blocks, threads, iters);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    *tflops = (float)(iter_flops * (double)iters * blocks * threads / (best * 1e-3) / 1e12);
    if (ms_out) *ms_out = best;
    return RT_OK;
}

extern "C" int rt_ffma_peak(rt_context *ctx, float *tflops, float *ms_out) {
    return peak_rate(ctx, 2.0 * 8 * 16, tflops, ms_out, [&](int blocks, int threads, int iters) {
        k_ffma_peak<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<float *>(ctx->counters.ptr), iters, 1.000001f, 1e-7f);
    });
}

// the same for packed half arithmetic: dense HFMA2 rate (2 lanes x 2 flop per instruction), the roofline denominator of USE_FP16
__global__ void __launch_bounds__(256) k_hfma2_peak(float *out, int iters, float a, float b) {
    const __half2 a2 = __float2half2_rn(a), b2 = __float2half2_rn(b);
    __half2 x[8];
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = __float2half2_rn((float)(threadIdx.x & 7) * 0.125f + (float)k);
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
#pragma unroll
            for (int k = 0; k < 8; k++) x[k] = __hfma2(x[k], a2, b2);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) s += __low2float(x[k]) + __high2float(x[k]);
    if (s == 12345.678f) out[0] = s;   // keeps the chain alive, never true in practice
}

extern "C" int rt_hfma2_peak(rt_context *ctx, float *tflops, float *ms_out) {
    return peak_rate(ctx, 4.0 * 8 * 16, tflops, ms_out, [&](int blocks, int threads, int iters) {
        k_hfma2_peak<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<float *>(ctx->counters.ptr), iters, 0.999f, 1e-3f);
    });
}

// ---- device memory helpers -----------------------------------------------------------------------------------------
extern "C" int rt_malloc(rt_context *ctx, size_t bytes, void **dev_ptr) {
    if (!ctx || !dev_ptr) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMalloc(dev_ptr, bytes));
    return RT_OK;
}
extern "C" int rt_free(rt_context *ctx, void *dev_ptr) {
    if (!ctx) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaFree(dev_ptr));
    return RT_OK;
}
extern "C" int rt_memcpy_to_host(rt_context *ctx, void *host, const void *dev, size_t bytes) {
    if (!ctx || !host || !dev) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}
extern "C" int rt_synchronize(rt_context *ctx) {
    if (!ctx) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// ---- multi-GPU: one context per GPU, one NCCL communicator over NVLink ------------------------------------------------
// The path has exactly one exchange (SURVEY §8e): the ranks' LINEAR radiance buffers are summed before /ns, sqrt and the
// output switch (main.cu:424-453).  NCCL is resolved at run time (dlopen) so that librt_b200.so has no link-time
// dependency and shares the NCCL already loaded in the process (torch's, in the Python host).
namespace {
struct NcclApi {
    void *handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclReduce) Reduce = nullptr;
    decltype(&ncclReduceScatter) ReduceScatter = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool ok = false;
};
NcclApi &nccl_api() {
    static NcclApi api = [] {
        NcclApi a;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            a.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (a.handle) break;
        }
        if (!a.handle) return a;
#define RT_NCCL_SYM(f) a.f = reinterpret_cast<decltype(a.f)>(dlsym(a.handle, "nccl" #f))
        RT_NCCL_SYM(GetUniqueId); RT_NCCL_SYM(CommInitRank); RT_NCCL_SYM(CommInitAll); RT_NCCL_SYM(CommDestroy); RT_NCCL_SYM(Reduce);
        RT_NCCL_SYM(ReduceScatter); RT_NCCL_SYM(Broadcast); RT_NCCL_SYM(GroupStart); RT_NCCL_SYM(GroupEnd); RT_NCCL_SYM(GetErrorString);
#undef RT_NCCL_SYM
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommInitAll && a.CommDestroy && a.Reduce && a.ReduceScatter && a.Broadcast &&
               a.GroupStart && a.GroupEnd && a.GetErrorString;
        return a;
    }();
    return api;
}
int nccl_fail(rt_context *ctx, ncclResult_t r, const char *what) {
    return fail(ctx, RT_ERR_STATE, "NCCL error %d at %s '%s'", (int)r, what, nccl_api().GetErrorString ? nccl_api().GetErrorString(r) : "?");
}
}  // namespace
#define NK(call)                                               \
    do {                                                       \
        ncclResult_t r_ = (call);                              \
        if (r_ != ncclSuccess) return nccl_fail(ctx, r_, #call); \
    } while (0)
#define NEED_NCCL(ctx) \
    if (!nccl_api().ok) return fail(ctx, RT_ERR_UNSUPPORTED, "libnccl.so.2 not found (or too old): multi-GPU entry points are unavailable")

static_assert(RT_COMM_ID_BYTES == sizeof(ncclUniqueId), "RT_COMM_ID_BYTES must match ncclUniqueId");

extern "C" int rt_comm_get_unique_id(void *id) {
    rt_context *ctx = nullptr;
    if (!id) return RT_ERR_INVALID;
    NEED_NCCL(ctx);
    NK(nccl_api().GetUniqueId(static_cast<ncclUniqueId *>(id)));
    return RT_OK;
}

extern "C" int rt_comm_init_rank(rt_context *ctx, const void *id, int nranks, int rank) {
    if (!ctx || !id || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, RT_ERR_INVALID, "rt_comm_init_rank: bad arguments");
    NEED_NCCL(ctx);
    if (ctx->comm) return fail(ctx, RT_ERR_STATE, "rt_comm_init_rank: the context already has a communicator");
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof uid);
    NK(nccl_api().CommInitRank(&ctx->comm, nranks, uid, rank));
    ctx->comm_owned = true; ctx->comm_rank = rank; ctx->comm_size = nranks;
    return RT_OK;
}

extern "C" int rt_comm_init_all(rt_context *const *ctxs, int n) {
    rt_context *ctx = (ctxs && n > 0) ? ctxs[0] : nullptr;
    if (!ctx || n > 64) return fail(ctx, RT_ERR_INVALID, "rt_comm_init_all: bad arguments");
    NEED_NCCL(ctx);
    int devs[64];
    ncclComm_t comms[64];
    for (int i = 0; i < n; i++) {
        if (!ctxs[i] || ctxs[i]->comm) return fail(ctx, RT_ERR_STATE, "rt_comm_init_all: null context, or one that already has a communicator");
        devs[i] = ctxs[i]->device;
    }
    NK(nccl_api().CommInitAll(comms, n, devs));
    for (int i = 0; i < n; i++) { ctxs[i]->comm = comms[i]; ctxs[i]->comm_owned = true; ctxs[i]->comm_rank = i; ctxs[i]->comm_size = n; }
    return RT_OK;
}

extern "C" int rt_comm_attach(rt_context *ctx, void *nccl_comm, int nranks, int rank) {
    if (!ctx || !nccl_comm || nranks < 1 || rank < 0 || rank >= nranks) return fail(ctx, RT_ERR_INVALID, "rt_comm_attach: bad arguments");
    NEED_NCCL(ctx);
    if (ctx->comm) return fail(ctx, RT_ERR_STATE, "rt_comm_attach: the context already has a communicator");
    ctx->comm = static_cast<ncclComm_t>(nccl_comm);
    ctx->comm_owned = false; ctx->comm_rank = rank; ctx->comm_size = nranks;
    return RT_OK;
}

extern "C" int rt_comm_destroy(rt_context *ctx) {
    if (!ctx) return RT_ERR_INVALID;
    if (ctx->comm && ctx->comm_owned) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        nccl_api().CommDestroy(ctx->comm);
    }
    ctx->comm = nullptr; ctx->comm_owned = false; ctx->comm_rank = 0; ctx->comm_size = 1;
    return RT_OK;
}

extern "C" int rt_comm_rank(const rt_context *ctx) { return ctx ? ctx->comm_rank : 0; }
extern "C" int rt_comm_size(const rt_context *ctx) { return ctx ? ctx->comm_size : 1; }

extern "C" int rt_group_start(void) { return nccl_api().ok && nccl_api().GroupStart() == ncclSuccess ? RT_OK : RT_ERR_STATE; }
extern "C" int rt_group_end(void) { return nccl_api().ok && nccl_api().GroupEnd() == ncclSuccess ? RT_OK : RT_ERR_STATE; }

extern "C" int rt_reduce(rt_context *ctx, float *accum_dev, size_t count, int root) {
    if (!ctx || !accum_dev) return fail(ctx, RT_ERR_INVALID, "rt_reduce: null argument");
    if (!ctx->comm) return ctx->comm_size == 1 ? RT_OK : fail(ctx, RT_ERR_STATE, "rt_reduce: no communicator (rt_comm_init_rank / rt_comm_init_all)");
    CK(cudaSetDevice(ctx->device));
    NK(nccl_api().Reduce(accum_dev, accum_dev, count, ncclFloat, ncclSum, root, ctx->comm, ctx->stream));
    return RT_OK;
}

extern "C" int rt_reduce_scatter(rt_context *ctx, const float *accum_dev, float *slice_dev, size_t slice_count) {
    if (!ctx || !accum_dev || !slice_dev) return fail(ctx, RT_ERR_INVALID, "rt_reduce_scatter: null argument");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->comm) {
        if (ctx->comm_size != 1) return fail(ctx, RT_ERR_STATE, "rt_reduce_scatter: no communicator");
        if (slice_dev != accum_dev) CK(cudaMemcpyAsync(slice_dev, accum_dev, slice_count * 4, cudaMemcpyDeviceToDevice, ctx->stream));
        return RT_OK;
    }
    NK(nccl_api().ReduceScatter(accum_dev, slice_dev, slice_count, ncclFloat, ncclSum, ctx->comm, ctx->stream));
    return RT_OK;
}

extern "C" int rt_broadcast(rt_context *ctx, void *dev, size_t bytes, int root) {
    if (!ctx || !dev) return fail(ctx, RT_ERR_INVALID, "rt_broadcast: null argument");
    if (!ctx->comm) return ctx->comm_size == 1 ? RT_OK : fail(ctx, RT_ERR_STATE, "rt_broadcast: no communicator");
    CK(cudaSetDevice(ctx->device));
    NK(nccl_api().Broadcast(dev, dev, bytes, ncclChar, root, ctx->comm, ctx->stream));
    return RT_OK;
}
