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
    bool slot0_defined = true;
    float4 *geom = nullptr, *matl = nullptr;
    int *tag = nullptr;
    size_t scene_cap = 0;
    // camera
    bool have_camera = false;
    int cam_nx = 0, cam_ny = 0;
    CameraData *cam_dev = nullptr;
    CameraData cam_host{};
    // octree
    OctreeBuilder *octree = nullptr;
    OctreeBuilder *list_accel = nullptr;     // USE_OCTREE off: the same grid over ALL spheres answers hitable_list::hit
    bool list_accel_valid = false;
    float grid_density = 4.0f;
    int default_variant = 0;       // RT_RENDER_VARIANT: kernel A/B override for whole test runs (0 = automatic)
    int last_kernel = 0;           // KernelId of the last render launch
    // render scratch
    uint32_t *work_counter = nullptr;
    unsigned long long *counters = nullptr;
    float *scratch_fb = nullptr;
    size_t scratch_fb_bytes = 0;
    PpmWorkspace ppm;
    float *pinned = nullptr;       // page-locked staging for the scene descriptors
    size_t pinned_bytes = 0;
    void *desc_dev = nullptr;      // ... and their raw device copy (split into geom / matl / tag by k_split_scene)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // RT_SEED_UPSTREAM: skip-ahead matrices (device copy) and the per-pixel stream states
    // RT_PREC_FP16: the scene rounded to half (8 B geometry + 8 B material per sphere) and the half camera
    uint2 *geom_h = nullptr, *matl_h = nullptr;
    size_t half_cap = 0;
    bool half_valid = false;
    HalfPairs half_pairs;
    __half *cam_h = nullptr;
    int cam_h_nx = 0, cam_h_ny = 0;
    rt_camera_desc cam_desc{};
    bool cam_desc_custom = false;
    uint32_t *skip_tables = nullptr;
    uint32_t *seed_states = nullptr;
    size_t seed_states_words = 0;
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
        (e = cudaMalloc(&ctx->work_counter, 4)) != cudaSuccess || (e = cudaMalloc(&ctx->counters, 32 * 8)) != cudaSuccess ||
        (e = cudaMalloc(&ctx->cam_dev, sizeof(CameraData))) != cudaSuccess) {
        delete ctx;
        return (int)e;
    }
    ctx->stream = ctx->own_stream;
    ctx->octree = new OctreeBuilder();
    ctx->list_accel = new OctreeBuilder();
    const char *dens = getenv("RT_GRID_DENSITY");
    if (dens && atof(dens) > 0) ctx->grid_density = (float)atof(dens);
    float flat = 0, wide = 0;
    unsigned flat_min = kFlatVoxelMinSpheres;
    const char *shape = getenv("RT_GRID_SHAPE");        // "flat:wide[:from how many spheres]", e.g. "1:1" for cubes everywhere
    if (shape && sscanf(shape, "%f:%f:%u", &flat, &wide, &flat_min) >= 2 && flat > 0 && wide > 0) {
        ctx->octree->grid_flat = ctx->list_accel->grid_flat = flat;
        ctx->octree->grid_wide = ctx->list_accel->grid_wide = wide;
        ctx->octree->grid_flat_min = ctx->list_accel->grid_flat_min = flat_min;
    }
    const char *var = getenv("RT_RENDER_VARIANT");
    if (var) ctx->default_variant = atoi(var);
    *out = ctx;
    return RT_OK;
}

extern "C" void rt_destroy(rt_context *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    delete ctx->octree;
    delete ctx->list_accel;
    ppm_free(ctx->ppm);
    cudaFree(ctx->geom); cudaFree(ctx->matl); cudaFree(ctx->tag); cudaFree(ctx->cam_dev);
    cudaFree(ctx->work_counter); cudaFree(ctx->counters); cudaFree(ctx->scratch_fb);
    cudaFree(ctx->skip_tables); cudaFree(ctx->seed_states);
    cudaFree(ctx->geom_h); cudaFree(ctx->matl_h); cudaFree(ctx->cam_h);
    cudaFree(ctx->half_pairs.geom); cudaFree(ctx->half_pairs.idx); cudaFree(ctx->half_pairs.start); cudaFree(ctx->half_pairs.count);
    cudaFree(ctx->half_pairs.nodes); cudaFree(ctx->half_pairs.node_count);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    cudaFree(ctx->desc_dev);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
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
    if ((size_t)n > ctx->scene_cap) {
        cudaFree(ctx->geom); cudaFree(ctx->matl); cudaFree(ctx->tag);
        ctx->geom = ctx->matl = nullptr; ctx->tag = nullptr; ctx->scene_cap = 0;
        CK(cudaMalloc(&ctx->geom, (size_t)n * sizeof(float4)));
        CK(cudaMalloc(&ctx->matl, (size_t)n * sizeof(float4)));
        CK(cudaMalloc(&ctx->tag, (size_t)n * sizeof(int)));
        ctx->scene_cap = (size_t)n;
    }
    const size_t bytes = (size_t)n * sizeof(rt_sphere_desc);
    CK(cudaStreamSynchronize(ctx->stream));                      // (an earlier upload may still be reading the staging buffer)
    if (bytes > ctx->pinned_bytes) {
        if (ctx->pinned) cudaFreeHost(ctx->pinned);
        ctx->pinned = nullptr; ctx->pinned_bytes = 0;
        cudaFree(ctx->desc_dev);
        ctx->desc_dev = nullptr;
        CK(cudaMallocHost(reinterpret_cast<void **>(&ctx->pinned), bytes + bytes / 4));
        ctx->pinned_bytes = bytes + bytes / 4;
        CK(cudaMalloc(&ctx->desc_dev, bytes + bytes / 4));
    }
    rt_sphere_desc *host = reinterpret_cast<rt_sphere_desc *>(ctx->pinned);
    memcpy(host, src, bytes);
    if (clamp_fuzz)
        for (int i = 0; i < n; i++)
            if (host[i].mat == RT_MAT_METAL && !(host[i].param < 1.0f)) host[i].param = 1.0f;   // metal::metal clamps fuzz (material.h:67)
    ctx->slot0_defined = host[0].mat != RT_MAT_NONE;
    CK(cudaMemcpyAsync(ctx->desc_dev, ctx->pinned, bytes, cudaMemcpyHostToDevice, ctx->stream));
    k_split_scene<<<(n + 255) / 256, 256, 0, ctx->stream>>>(static_cast<const rt_sphere_desc *>(ctx->desc_dev), n, ctx->geom, ctx->matl, ctx->tag);
    CK(cudaGetLastError());
    ctx->octree->built = false;
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
    memcpy(out, ctx->pinned, (size_t)n * sizeof(rt_sphere_desc));      // the staging buffer of the last upload
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
    k_camera_setup<<<1, 1, 0, ctx->stream>>>(c, ctx->cam_dev);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(&ctx->cam_host, ctx->cam_dev, sizeof(CameraData), cudaMemcpyDeviceToHost, ctx->stream));
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
    if (!ctx->cam_h) CK(cudaMalloc(&ctx->cam_h, 22 * sizeof(__half)));
    if (ctx->cam_h_nx != nx || ctx->cam_h_ny != ny) {
        const rt_camera_desc &c = ctx->cam_desc;
        CK(launch_camera_setup_half(c.lookfrom, c.lookat, c.vup, c.vfov, nx, ny, ctx->cam_desc_custom ? c.aspect : 0.f, c.aperture,
                                    c.focus_dist, ctx->cam_h, ctx->stream));
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
    CK(cudaMemcpyAsync(h, ctx->cam_h, sizeof h, cudaMemcpyDeviceToHost, ctx->stream));
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
    CK(ctx->octree->build(ctx->stream, ctx->geom, ctx->tag, ctx->n, spl, ctx->grid_density, precision == RT_PREC_FP16));
    ctx->half_pairs.valid = false;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaEventSynchronize(ctx->ev1));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        stats->build_ms = ms;
        stats->node_count = ctx->octree->counts.node_count;
        stats->entries = (int64_t)ctx->octree->stats_h[0];
        stats->dropped_full = (int64_t)ctx->octree->stats_h[1];
        stats->dropped_outside = (int64_t)ctx->octree->stats_h[2];
        stats->fine_voxels = ctx->octree->total_voxels;
        stats->fine_refs = ctx->octree->total_refs;
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
    if (!ctx->octree->built) return fail(ctx, RT_ERR_STATE, "rt_octree_export_reference: build the octree first");
    if (ctx->octree->fp16) {      // the USE_FP16 AABB holds the planes as halves: they must be exact there (k_blob_nodes)
        const float *pl = &ctx->octree->planes.p[0][0];
        for (int k = 0; k < 3 * kPlanes; k++)
            if (__half2float(__float2half_rn(pl[k])) != pl[k])
                return fail(ctx, RT_ERR_UNSUPPORTED, "rt_octree_export_reference: box plane %g is not exact in half", (double)pl[k]);
    }
    CK(cudaSetDevice(ctx->device));
    CK(ctx->octree->export_reference(ctx->stream, host_blob, bytes));
    return RT_OK;
}

extern "C" size_t rt_octree_debug_read(rt_context *ctx, int which, void *host, size_t cap) {
    if (!ctx) return 0;
    cudaSetDevice(ctx->device);
    return ctx->octree->debug_read(ctx->stream, which, host, cap);
}

// ---- USE_FP16 state -------------------------------------------------------------------------------------------------
// What the half kernels read, derived on demand and kept until the scene, the tree or the frame size changes: always the scene
// rounded to half; with kHalfPairs the pair lists of one mode (octree: the cells of `tv`; flat: all spheres); with kHalfCamera
// the half camera of an nx x ny frame.  The render and the per-ray entry points share it.
enum { kHalfPairs = 1, kHalfCamera = 2 };
static int ensure_half(rt_context *ctx, unsigned what, bool octree, const TreeView &tv, int nx, int ny) {
    if (ctx->half_cap < (size_t)ctx->n) {
        cudaFree(ctx->geom_h); cudaFree(ctx->matl_h);
        ctx->geom_h = ctx->matl_h = nullptr; ctx->half_cap = 0;
        CK(cudaMalloc(&ctx->geom_h, (size_t)ctx->n * sizeof(uint2)));
        CK(cudaMalloc(&ctx->matl_h, (size_t)ctx->n * sizeof(uint2)));
        ctx->half_cap = (size_t)ctx->n;
        ctx->half_valid = false;
    }
    if (!ctx->half_valid) {
        CK(launch_scene_to_half(ctx->geom, ctx->matl, ctx->n, ctx->geom_h, ctx->matl_h, ctx->stream));
        ctx->half_valid = true;
        ctx->half_pairs.valid = false;
    }
    if ((what & kHalfPairs) && (!ctx->half_pairs.valid || ctx->half_pairs.octree != octree))
        CK(build_half_pairs(ctx->half_pairs, ctx->geom_h, ctx->tag, ctx->n, octree, tv, ctx->stream));
    if (what & kHalfCamera) return ensure_half_camera(ctx, nx, ny);
    return RT_OK;
}

// ---- render -----------------------------------------------------------------------------------------------------
struct ProgressiveIO {
    uint32_t *state = nullptr;     // 6 words per pixel, device
    bool first = true;
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
static int do_render(rt_context *ctx, const rt_render_args *a, float *out_dev, bool finalize, rt_render_stats *stats,
                     const ProgressiveIO *prog = nullptr, const PixelList *list = nullptr) {
    if (!ctx || !a || !out_dev) return fail(ctx, RT_ERR_INVALID, "render: null argument");
    if (a->nx < 1 || a->ny < 1 || a->ns < 1) return fail(ctx, RT_ERR_INVALID, "render: bad nx/ny/ns");
    if (list) {
        if (!list->pixels || list->count < 1) return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: null pixel list or count < 1");
        if (a->shard_mode != RT_SHARD_NONE) return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: pixel lists are not sharded (give each GPU its own list)");
        if (!on_device(ctx, list->pixels) || !on_device(ctx, out_dev))
            return fail(ctx, RT_ERR_INVALID, "rt_render_pixels: pixels_dev and out_dev must be device memory of the context's GPU");
    }
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "render: no scene (rt_scene_generate / rt_scene_upload first)");
    if (a->use_octree && !ctx->octree->built) return fail(ctx, RT_ERR_STATE, "render: USE_OCTREE set but no octree built");
    if (a->seed_mode != RT_SEED_HEAD && a->seed_mode != RT_SEED_UPSTREAM) return fail(ctx, RT_ERR_INVALID, "render: unknown seed_mode");
    if (a->precision != RT_PREC_FP32 && a->precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "render: unknown precision");
    const bool fp16 = a->precision == RT_PREC_FP16;
    // a tile shard holds whole pixels' half sums, exact in float, so shards add up to the 1-GPU frame; the half sum of ns/G
    // samples per rank is a different image from any build of the reference
    if (fp16 && a->shard_mode == RT_SHARD_SPP)
        return fail(ctx, RT_ERR_UNSUPPORTED, "render: USE_FP16 frames shard by tiles only (RT_SHARD_TILES): spp shards' half sums do not add up to the 1-GPU frame");
    if (a->use_octree && ctx->octree->built && ctx->octree->fp16 != fp16)
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
    p.scene.geom = ctx->geom; p.scene.matl = ctx->matl; p.scene.tag = ctx->tag; p.scene.n = ctx->n;
    if (a->use_octree) p.tree = ctx->octree->view();
    // flat-list mode: hitable_list::hit is "closest over all spheres"; above a few hundred spheres the grid answers it
    // with a few dozen tests instead of N (the result is the same minimum; variant 20 forces the N-test sweep)
    bool list_grid = false;
    if (!a->use_octree && a->precision == RT_PREC_FP32 && ctx->n >= kListGridMinSpheres && a->tune[1] != 20 &&
        ctx->slot0_defined) {      // (the prolog tests sphere 0 unconditionally; an undefined slot 0 must stay unhittable)
        if (!ctx->list_accel_valid) {
            CK(ctx->list_accel->build(ctx->stream, ctx->geom, ctx->tag, ctx->n, 30, ctx->grid_density, false, true));
            ctx->list_accel_valid = true;
        }
        p.tree = ctx->list_accel->view();
        list_grid = true;
    }
    p.cam = ctx->cam_host;                        // per-context camera, by value in the launch parameters
    {
        const OctreeBuilder *acc = list_grid ? ctx->list_accel : ctx->octree;
        p.coop_items = (a->use_octree || list_grid) && acc->total_voxels > 0 && acc->total_refs / acc->total_voxels >= 40 ? 4 : 2;
    }
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
    p.total_items = list ? (uint32_t)list->count : (uint32_t)(owned * 32);
    if (list) p.pixels = list->pixels;
    p.finalize = finalize ? 1 : 0;
    p.variant = a->tune[1] ? a->tune[1] : ctx->default_variant;
    p.out = out_dev;
    p.work_counter = ctx->work_counter;
    p.counters = ctx->counters;
    CK(cudaMemsetAsync(ctx->counters, 0, 32 * 8, ctx->stream));
    int blocks = 0;
    int launches = 1;
    if (a->seed_mode == RT_SEED_UPSTREAM && !continuing) {
        const size_t npix = list ? (size_t)list->count : (size_t)a->nx * a->ny;      // stream states to seed
        if (!ctx->skip_tables) {
            const std::vector<uint32_t> &t = host_skip_tables();
            CK(cudaMalloc(&ctx->skip_tables, t.size() * 4));
            CK(cudaMemcpyAsync(ctx->skip_tables, t.data(), t.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
        }
        if (ctx->seed_states_words < npix * 6) {
            cudaFree(ctx->seed_states);
            ctx->seed_states = nullptr; ctx->seed_states_words = 0;
            CK(cudaMalloc(&ctx->seed_states, npix * 6 * 4));
            ctx->seed_states_words = npix * 6;
        }
        p.seed_states = ctx->seed_states;
    }
    if (prog) {
        p.state_out = prog->state;
        p.accumulate = continuing ? 1 : 0;
    }
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (continuing) {
        p.seed_states = prog->state;                  // every pixel resumes its own stream
    } else if (p.seed_states) {   // render_init (main.cu:424): inside the timed region, as in the reference
        if (list)                 // only the listed pixels' streams
            CK(launch_seed_upstream_list(ctx->seed_states, list->pixels, list->count, (size_t)a->nx * a->ny, 1984ull, ctx->skip_tables,
                                         ctx->stream));
        else                      // spp shard g draws from subsequences pixel_index + g * num_pixels (g = 0: the reference's streams)
            CK(launch_seed_upstream(ctx->seed_states, (size_t)a->nx * a->ny, 1984ull, p.seed_offset, ctx->skip_tables, ctx->stream));
        launches = 2;
    }
    if (fp16) {
        {
            const int rc = ensure_half(ctx, kHalfPairs | kHalfCamera, a->use_octree != 0, p.tree, a->nx, a->ny);
            if (rc) return rc;
        }
        CK(launch_render_half(p, a->use_octree != 0, ctx->geom_h, ctx->matl_h, ctx->cam_h, ctx->half_pairs, ctx->prop.multiProcessorCount,
                              ctx->stream, &blocks, list != nullptr));
        ctx->last_kernel = kKernelHalf;
    } else {
        CK(launch_render(p, a->use_octree != 0 || list_grid, ctx->prop.multiProcessorCount, ctx->prop.sharedMemPerBlockOptin, ctx->stream, &blocks,
                         &ctx->last_kernel, list != nullptr));
    }
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    if (stats) {
        unsigned long long c[4] = {0, 0, 0, 0};
        CK(cudaMemcpyAsync(c, ctx->counters, sizeof c, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        CK(cudaStreamSynchronize(ctx->stream));
        memset(stats, 0, sizeof *stats);
        stats->rays = c[0]; stats->paths = c[1];
        stats->sphere_tests = c[2]; stats->node_tests = c[3];   // zero unless built with -DRT_COUNTERS
        stats->kernel_id = ctx->last_kernel;
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        stats->kernel_ms = ms;
        stats->launches = launches;
    }
    return RT_OK;
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
    unsigned long long c[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(c, ctx->counters, sizeof c, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    memset(stats, 0, sizeof *stats);
    stats->rays = c[0]; stats->paths = c[1];
    stats->sphere_tests = c[2]; stats->node_tests = c[3];
    stats->kernel_id = ctx->last_kernel;
    stats->launches = 1;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) == cudaSuccess) stats->kernel_ms = ms;
    return RT_OK;
}

// test hook: the raw device counters of the last render
extern "C" int rt_debug_counters(rt_context *ctx, uint64_t out[32]) {
    if (!ctx || !out) return fail(ctx, RT_ERR_INVALID, "rt_debug_counters: null argument");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(out, ctx->counters, 32 * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// device scratch of one API call, released on every exit path
struct Scratch {
    std::vector<void *> ptrs;
    ~Scratch() { for (void *p : ptrs) cudaFree(p); }
    template <typename T>
    cudaError_t get(T *&out, size_t count) {
        void *p = nullptr;
        const cudaError_t e = cudaMalloc(&p, count * sizeof(T) + 16);
        if (e == cudaSuccess) ptrs.push_back(p);
        out = static_cast<T *>(p);
        return e;
    }
};

// test hook: closest hit of caller-supplied rays (host arrays of 3 floats per ray)
extern "C" int rt_trace_rays(rt_context *ctx, int use_octree, int n, const float *org, const float *dir, int *out_idx, float *out_t) {
    if (!ctx || n < 1 || !org || !dir || !out_idx || !out_t) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_trace_rays: no scene");
    if (use_octree && !ctx->octree->built) return fail(ctx, RT_ERR_STATE, "rt_trace_rays: no octree built");
    CK(cudaSetDevice(ctx->device));
    Scratch sc;
    float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr;
    int *d_i = nullptr;
    CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3));
    CK(sc.get(d_t, (size_t)n)); CK(sc.get(d_i, (size_t)n));
    CK(cudaMemcpyAsync(d_o, org, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_d, dir, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    RenderLaunch p;
    memset(&p, 0, sizeof p);
    p.scene.geom = ctx->geom; p.scene.matl = ctx->matl; p.scene.tag = ctx->tag; p.scene.n = ctx->n;
    if (use_octree) p.tree = ctx->octree->view();
    p.variant = ctx->default_variant;
    CK(launch_trace_rays(p, use_octree != 0, d_o, d_d, n, d_i, d_t, ctx->stream));
    CK(cudaMemcpyAsync(out_idx, d_i, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_t, d_t, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// camera::get_ray (camera.h:45-49) for n (s, t) pairs: each draws its lens sample from ITS OWN XORWOW state (6 words, in/out)
extern "C" int rt_camera_get_rays(rt_context *ctx, int n, const float *s, const float *t, uint32_t *states6, float *org, float *dir) {
    if (!ctx || n < 1 || !s || !t || !states6 || !org || !dir) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_rays: bad arguments");
    if (!ctx->have_camera) return fail(ctx, RT_ERR_STATE, "rt_camera_get_rays: no camera set (rt_camera_set)");
    CK(cudaSetDevice(ctx->device));
    Scratch sc;
    float *d_s = nullptr, *d_t = nullptr, *d_o = nullptr, *d_d = nullptr;
    uint32_t *d_st = nullptr;
    CK(sc.get(d_s, (size_t)n)); CK(sc.get(d_t, (size_t)n)); CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3)); CK(sc.get(d_st, (size_t)n * 6));
    CK(cudaMemcpyAsync(d_s, s, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_t, t, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_st, states6, (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_camera_rays(ctx->cam_host, n, d_s, d_t, d_st, d_o, d_d, ctx->stream));
    CK(cudaMemcpyAsync(org, d_o, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dir, d_d, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(states6, d_st, (size_t)n * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// material::scatter (material.h:55-113) + the hit record of sphere::hit (sphere.h:30-33) for n (ray, sphere, t) triples
extern "C" int rt_scatter_rays(rt_context *ctx, int n, const int *sphere_idx, const float *org, const float *dir, const float *t_hit,
                               uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten, int *scattered) {
    if (!ctx || n < 1 || !sphere_idx || !org || !dir || !t_hit || !states6 || !out_p || !out_normal || !out_dir || !out_atten || !scattered)
        return fail(ctx, RT_ERR_INVALID, "rt_scatter_rays: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_scatter_rays: no scene");
    CK(cudaSetDevice(ctx->device));
    Scratch sc;
    int *d_i = nullptr, *d_sc = nullptr;
    float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr, *d_p = nullptr, *d_n = nullptr, *d_od = nullptr, *d_a = nullptr;
    uint32_t *d_st = nullptr;
    CK(sc.get(d_i, (size_t)n)); CK(sc.get(d_sc, (size_t)n)); CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3)); CK(sc.get(d_t, (size_t)n));
    CK(sc.get(d_p, (size_t)n * 3)); CK(sc.get(d_n, (size_t)n * 3)); CK(sc.get(d_od, (size_t)n * 3)); CK(sc.get(d_a, (size_t)n * 3)); CK(sc.get(d_st, (size_t)n * 6));
    CK(cudaMemcpyAsync(d_i, sphere_idx, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_o, org, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_d, dir, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_t, t_hit, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_st, states6, (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_p, 0, (size_t)n * 12, ctx->stream)); CK(cudaMemsetAsync(d_n, 0, (size_t)n * 12, ctx->stream));
    CK(cudaMemsetAsync(d_od, 0, (size_t)n * 12, ctx->stream)); CK(cudaMemsetAsync(d_a, 0, (size_t)n * 12, ctx->stream));
    SceneView sv;
    sv.geom = ctx->geom; sv.matl = ctx->matl; sv.tag = ctx->tag; sv.n = ctx->n;
    CK(launch_scatter_rays(sv, n, d_i, d_o, d_d, d_t, d_st, d_p, d_n, d_od, d_a, d_sc, ctx->stream));
    CK(cudaMemcpyAsync(out_p, d_p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_normal, d_n, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_dir, d_od, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_atten, d_a, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(scattered, d_sc, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(states6, d_st, (size_t)n * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

// ---- the same three queries under a given arithmetic ----------------------------------------------------------------------
// RT_PREC_FP16: the USE_FP16 build's hitTree / hitable_list::hit, camera::get_ray and material::scatter (rt_render_half.cuh):
// float inputs are rounded to half on entry, outputs are halves widened to float.
extern "C" int rt_trace_rays_ex(rt_context *ctx, int use_octree, int precision, int n, const float *org, const float *dir, int *out_idx,
                                float *out_t) {
    if (precision != RT_PREC_FP32 && precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays_ex: unknown precision");
    if (!ctx || n < 1 || !org || !dir || !out_idx || !out_t) return fail(ctx, RT_ERR_INVALID, "rt_trace_rays_ex: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: no scene");
    if (use_octree && !ctx->octree->built) return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: no octree built");
    if (use_octree && ctx->octree->fp16 != (precision == RT_PREC_FP16))
        return fail(ctx, RT_ERR_STATE, "rt_trace_rays_ex: the octree was built for the other precision (rt_octree_build_ex)");
    if (precision == RT_PREC_FP32) return rt_trace_rays(ctx, use_octree, n, org, dir, out_idx, out_t);
    CK(cudaSetDevice(ctx->device));
    RenderLaunch p;
    memset(&p, 0, sizeof p);
    p.scene.geom = ctx->geom; p.scene.matl = ctx->matl; p.scene.tag = ctx->tag; p.scene.n = ctx->n;
    if (use_octree) p.tree = ctx->octree->view();
    {
        const int rc = ensure_half(ctx, kHalfPairs, use_octree != 0, p.tree, 0, 0);
        if (rc) return rc;
    }
    Scratch sc;
    float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr;
    int *d_i = nullptr;
    CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3));
    CK(sc.get(d_t, (size_t)n)); CK(sc.get(d_i, (size_t)n));
    CK(cudaMemcpyAsync(d_o, org, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_d, dir, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_trace_rays_half(p, use_octree != 0, ctx->geom_h, ctx->half_pairs, d_o, d_d, n, d_i, d_t, ctx->stream));
    CK(cudaMemcpyAsync(out_idx, d_i, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_t, d_t, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

extern "C" int rt_camera_get_rays_ex(rt_context *ctx, int precision, int n, const float *s, const float *t, uint32_t *states6, float *org,
                                     float *dir) {
    if (precision == RT_PREC_FP32) return rt_camera_get_rays(ctx, n, s, t, states6, org, dir);
    if (precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_rays_ex: unknown precision");
    if (!ctx || n < 1 || !s || !t || !states6 || !org || !dir) return fail(ctx, RT_ERR_INVALID, "rt_camera_get_rays_ex: bad arguments");
    if (!ctx->have_camera) return fail(ctx, RT_ERR_STATE, "rt_camera_get_rays_ex: no camera set (rt_camera_set)");
    CK(cudaSetDevice(ctx->device));
    {
        const int rc = ensure_half_camera(ctx, ctx->cam_nx, ctx->cam_ny);      // the camera the FP16 render of this frame size uses
        if (rc) return rc;
    }
    Scratch sc;
    float *d_s = nullptr, *d_t = nullptr, *d_o = nullptr, *d_d = nullptr;
    uint32_t *d_st = nullptr;
    CK(sc.get(d_s, (size_t)n)); CK(sc.get(d_t, (size_t)n)); CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3)); CK(sc.get(d_st, (size_t)n * 6));
    CK(cudaMemcpyAsync(d_s, s, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_t, t, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_st, states6, (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream));
    CK(launch_camera_rays_half(ctx->cam_h, n, d_s, d_t, d_st, d_o, d_d, ctx->stream));
    CK(cudaMemcpyAsync(org, d_o, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(dir, d_d, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(states6, d_st, (size_t)n * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

extern "C" int rt_scatter_rays_ex(rt_context *ctx, int precision, int n, const int *sphere_idx, const float *org, const float *dir,
                                  const float *t_hit, uint32_t *states6, float *out_p, float *out_normal, float *out_dir, float *out_atten,
                                  int *scattered) {
    if (precision == RT_PREC_FP32)
        return rt_scatter_rays(ctx, n, sphere_idx, org, dir, t_hit, states6, out_p, out_normal, out_dir, out_atten, scattered);
    if (precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_scatter_rays_ex: unknown precision");
    if (!ctx || n < 1 || !sphere_idx || !org || !dir || !t_hit || !states6 || !out_p || !out_normal || !out_dir || !out_atten || !scattered)
        return fail(ctx, RT_ERR_INVALID, "rt_scatter_rays_ex: bad arguments");
    if (ctx->n < 1) return fail(ctx, RT_ERR_STATE, "rt_scatter_rays_ex: no scene");
    CK(cudaSetDevice(ctx->device));
    {
        const TreeView none{};
        const int rc = ensure_half(ctx, 0u, false, none, 0, 0);
        if (rc) return rc;
    }
    Scratch sc;
    int *d_i = nullptr, *d_sc = nullptr;
    float *d_o = nullptr, *d_d = nullptr, *d_t = nullptr, *d_p = nullptr, *d_n = nullptr, *d_od = nullptr, *d_a = nullptr;
    uint32_t *d_st = nullptr;
    CK(sc.get(d_i, (size_t)n)); CK(sc.get(d_sc, (size_t)n)); CK(sc.get(d_o, (size_t)n * 3)); CK(sc.get(d_d, (size_t)n * 3)); CK(sc.get(d_t, (size_t)n));
    CK(sc.get(d_p, (size_t)n * 3)); CK(sc.get(d_n, (size_t)n * 3)); CK(sc.get(d_od, (size_t)n * 3)); CK(sc.get(d_a, (size_t)n * 3)); CK(sc.get(d_st, (size_t)n * 6));
    CK(cudaMemcpyAsync(d_i, sphere_idx, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_o, org, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_d, dir, (size_t)n * 12, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_t, t_hit, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_st, states6, (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemsetAsync(d_p, 0, (size_t)n * 12, ctx->stream)); CK(cudaMemsetAsync(d_n, 0, (size_t)n * 12, ctx->stream));
    CK(cudaMemsetAsync(d_od, 0, (size_t)n * 12, ctx->stream)); CK(cudaMemsetAsync(d_a, 0, (size_t)n * 12, ctx->stream));
    SceneView sv;
    sv.geom = ctx->geom; sv.matl = ctx->matl; sv.tag = ctx->tag; sv.n = ctx->n;
    CK(launch_scatter_rays_half(sv, ctx->geom_h, ctx->matl_h, n, d_i, d_o, d_d, d_t, d_st, d_p, d_n, d_od, d_a, d_sc, ctx->stream));
    CK(cudaMemcpyAsync(out_p, d_p, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_normal, d_n, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_dir, d_od, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_atten, d_a, (size_t)n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(scattered, d_sc, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(states6, d_st, (size_t)n * 24, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
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

extern "C" int rt_render_progressive(rt_context *ctx, const rt_render_args *args, float *accum_dev, uint32_t *rng_state_dev, int first,
                                     rt_render_stats *stats) {
    if (!rng_state_dev) return fail(ctx, RT_ERR_INVALID, "rt_render_progressive: null state buffer");
    ProgressiveIO io;
    io.state = rng_state_dev;
    io.first = first != 0;
    return do_render(ctx, args, accum_dev, false, stats, &io);
}

extern "C" int rt_finalize(rt_context *ctx, const float *accum_dev, float *fb_dev, int nx, int ny, int ns) {
    if (!ctx || !accum_dev || !fb_dev || nx < 1 || ny < 1 || ns < 1) return fail(ctx, RT_ERR_INVALID, "rt_finalize: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(launch_finalize(accum_dev, fb_dev, nx, ny, ns, ctx->stream));
    return RT_OK;
}

extern "C" int rt_finalize_n(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns) {
    if (!ctx || !accum_dev || !fb_dev || ns < 1) return fail(ctx, RT_ERR_INVALID, "rt_finalize_n: bad arguments");
    if (count == 0) return RT_OK;
    CK(cudaSetDevice(ctx->device));
    CK(launch_finalize_n(accum_dev, fb_dev, count, ns, ctx->stream));
    return RT_OK;
}

extern "C" int rt_finalize_ex(rt_context *ctx, const float *accum_dev, float *fb_dev, size_t count, int ns, int precision) {
    if (precision == RT_PREC_FP32) return rt_finalize_n(ctx, accum_dev, fb_dev, count, ns);
    if (precision != RT_PREC_FP16) return fail(ctx, RT_ERR_INVALID, "rt_finalize_ex: unknown precision");
    if (!ctx || !accum_dev || !fb_dev || ns < 1) return fail(ctx, RT_ERR_INVALID, "rt_finalize_ex: bad arguments");
    if (count == 0) return RT_OK;
    CK(cudaSetDevice(ctx->device));
    CK(launch_finalize_half(accum_dev, fb_dev, count, ns, ctx->stream));
    return RT_OK;
}

extern "C" int rt_render_to_host(rt_context *ctx, const rt_render_args *args, float *fb_host, rt_render_stats *stats) {
    if (!ctx || !args || !fb_host) return fail(ctx, RT_ERR_INVALID, "rt_render_to_host: null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)args->nx * args->ny * 3 * sizeof(float);
    if (bytes > ctx->scratch_fb_bytes) {
        cudaFree(ctx->scratch_fb);
        ctx->scratch_fb = nullptr; ctx->scratch_fb_bytes = 0;
        CK(cudaMalloc(&ctx->scratch_fb, bytes));
        ctx->scratch_fb_bytes = bytes;
    }
    const int rc = do_render(ctx, args, ctx->scratch_fb, true, stats);
    if (rc) return rc;
    CK(cudaMemcpyAsync(fb_host, ctx->scratch_fb, bytes, cudaMemcpyDeviceToHost, ctx->stream));
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
    if (!ctx->ppm.text || cap < ctx->ppm.text_len) return fail(ctx, RT_ERR_INVALID, "rt_ppm_read: no formatted frame, or the buffer is smaller than its text");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpyAsync(buf_host, ctx->ppm.text, ctx->ppm.text_len, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RT_OK;
}

extern "C" int rt_render_to_ppm(rt_context *ctx, const rt_render_args *args, rt_render_stats *stats, size_t *len_out) {
    if (!ctx || !args) return fail(ctx, RT_ERR_INVALID, "rt_render_to_ppm: null argument");
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)args->nx * args->ny * 3 * sizeof(float);
    if (bytes > ctx->scratch_fb_bytes) {
        cudaFree(ctx->scratch_fb);
        ctx->scratch_fb = nullptr; ctx->scratch_fb_bytes = 0;
        CK(cudaMalloc(&ctx->scratch_fb, bytes));
        ctx->scratch_fb_bytes = bytes;
    }
    const int rc = do_render(ctx, args, ctx->scratch_fb, true, stats);
    if (rc) return rc;
    CK(ppm_format_device(ctx->ppm, ctx->scratch_fb, args->nx, args->ny, ctx->stream, len_out));
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

extern "C" int rt_ffma_peak(rt_context *ctx, float *tflops, float *ms_out) {
    if (!ctx || !tflops) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        k_ffma_peak<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<float *>(ctx->counters), iters, 1.000001f, 1e-7f);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    const double flops = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    *tflops = (float)(flops / (best * 1e-3) / 1e12);
    if (ms_out) *ms_out = best;
    return RT_OK;
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
    if (!ctx || !tflops) return RT_ERR_INVALID;
    CK(cudaSetDevice(ctx->device));
    const int blocks = ctx->prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        k_hfma2_peak<<<blocks, threads, 0, ctx->stream>>>(reinterpret_cast<float *>(ctx->counters), iters, 0.999f, 1e-3f);
        CK(cudaEventRecord(ctx->ev1, ctx->stream));
        CK(cudaEventSynchronize(ctx->ev1));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    const double flops = 4.0 * 8 * 16 * (double)iters * blocks * threads;
    *tflops = (float)(flops / (best * 1e-3) / 1e12);
    if (ms_out) *ms_out = best;
    return RT_OK;
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
