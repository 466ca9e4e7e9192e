// raytracing_main.cpp — the reference's CLI, `RayTracing [mode]` (main.cu:347-477), over the C ABI.
//
//   mode 0 = P3 PPM to stdout (default), 1 = no output, 3 = output.ppm; 2 (OpenGL preview) is accepted and ignored.
// Same banner on stderr, same "took X seconds." line, same exit(99) on a CUDA error.  The reference's knobs keep
// their names; they are #ifndef-guarded so -D works, and can be overridden at run time without touching the
// positional argument: RT_NUM_SPHERES, RT_SPHERES_PER_LEAF, RT_USE_OCTREE, RT_USE_FP16, RT_NX, RT_NY, RT_NS
// (and RT_SEED_MODE=1 for the upstream per-pixel seeding curand_init(1984, pixel_index, 0), main.cu:90).
// RT_GPUS=N shards the frame over N GPUs of this box (one context per GPU, rt_comm_* / rt_reduce: NCCL over NVLink);
// RT_SHARD=tiles (default, bit-identical to one GPU) or spp; USE_FP16 frames shard by tiles only.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include "rt_abi.h"

#ifndef NUM_SPHERES
#define NUM_SPHERES 8000          // main.cu:22
#endif
#ifndef SPHERE_RADIUS
#define SPHERE_RADIUS 0.1f        // main.cu:23
#endif
#ifndef SPHERES_PER_LEAF
#define SPHERES_PER_LEAF 30       // acceleration_structure.h:15
#endif
#ifndef RT_NO_OCTREE
#define USE_OCTREE                // main.cu:24
#endif

static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// check_cuda (main.cu:29-37): message, then exit(99)
static void check(rt_context *ctx, int rc, const char *what, const char *file, int line) {
    if (rc) {
        std::cerr << "CUDA error = " << static_cast<unsigned int>(rc) << " at " << file << ":" << line << " '" << what << "' \n";
        if (ctx) std::cerr << rt_last_error(ctx) << "\n";
        exit(99);
    }
}
#define CHECK(call) check(ctx, (call), #call, __FILE__, __LINE__)

int main(int argc, char **argv) {
    const int nx = env_int("RT_NX", 1200), ny = env_int("RT_NY", 800), ns = env_int("RT_NS", 10);   // main.cu:348-350
    const int tx = 8, ty = 8;
    const int n = env_int("RT_NUM_SPHERES", NUM_SPHERES);
    const int spl = env_int("RT_SPHERES_PER_LEAF", SPHERES_PER_LEAF);
#ifdef USE_OCTREE
    const int use_octree = env_int("RT_USE_OCTREE", 1);
#else
    const int use_octree = env_int("RT_USE_OCTREE", 0);
#endif
    std::cerr << "Rendering a " << nx << "x" << ny << " image with " << ns << " samples per pixel ";
    std::cerr << "in " << tx << "x" << ty << " blocks.\n";
    std::cerr << "Number of spheres: " << n << "\n";
    std::cerr << "Sphere radius: " << SPHERE_RADIUS << "\n";
    std::cerr << (use_octree ? "Use octree: ON\n" : "Use octree: OFF\n");
#ifdef USE_FP16                   // precision_types.h:8
    const int precision = env_int("RT_USE_FP16", 1) ? RT_PREC_FP16 : RT_PREC_FP32;
#else
    const int precision = env_int("RT_USE_FP16", 0) ? RT_PREC_FP16 : RT_PREC_FP32;
#endif
    int output_mode = 0;
    if (argc > 1) output_mode = std::stoi(argv[1]);      // throws on garbage, as the reference does
    std::cerr << "Output mode: " << output_mode << "\n";

    const int gpus = env_int("RT_GPUS", 1);             // > 1: the frame is sharded over that many GPUs of this box (NCCL reduce)
    rt_render_args a{};
    a.nx = nx; a.ny = ny; a.ns = ns; a.max_depth = 50; a.use_octree = use_octree;
    a.precision = precision;
    a.seed_mode = env_int("RT_SEED_MODE", RT_SEED_HEAD);
    const size_t n3 = (size_t)nx * ny * 3;
    const bool want_text = output_mode == 0 || output_mode == 3;
    std::vector<float> fb_host;
    size_t need = 0;
    rt_context *ctx = nullptr;                           // the context that ends up holding the frame (rank 0)
    std::vector<rt_context *> ctxs((size_t)(gpus > 1 ? gpus : 1), nullptr);
    std::vector<float *> bufs(ctxs.size(), nullptr);
    double secs = 0;
    rt_render_stats st{};

    // world + octree + camera on every GPU (main.cu:388-415), in parallel
    {
        std::vector<std::thread> th;
        std::vector<int> rcs(ctxs.size(), 0);
        for (size_t g = 0; g < ctxs.size(); g++)
            th.emplace_back([&, g] {
                int rc = rt_create((int)g, &ctxs[g]);
                if (!rc) rc = rt_scene_generate_ex(ctxs[g], n, SPHERE_RADIUS, precision);
                if (!rc && use_octree) rc = rt_octree_build_ex(ctxs[g], spl, precision, nullptr);
                if (!rc) rc = rt_camera_set(ctxs[g], nullptr, nx, ny);
                if (!rc) rc = rt_malloc(ctxs[g], n3 * sizeof(float), reinterpret_cast<void **>(&bufs[g]));
                rcs[g] = rc;
            });
        for (auto &t : th) t.join();
        for (size_t g = 0; g < ctxs.size(); g++) { ctx = ctxs[g]; CHECK(rcs[g]); }
        ctx = ctxs[0];
    }
    if (gpus > 1) {
        // RT_SHARD=tiles (default): interleaved 8x4 tiles, the summed frame is bit-identical to the 1-GPU frame;
        // RT_SHARD=spp: every GPU traces ns/gpus samples of every pixel from its own streams (better balance, same quality)
        const char *sh = getenv("RT_SHARD");
        a.shard_mode = sh && std::string(sh) == "spp" ? RT_SHARD_SPP : RT_SHARD_TILES;
        if (precision == RT_PREC_FP16 && a.shard_mode == RT_SHARD_SPP) {
            std::cerr << "USE_FP16 frames shard by tiles only (RT_SHARD=tiles): spp shards' half sums do not add up to the 1-GPU frame\n";
            exit(99);
        }
        CHECK(rt_comm_init_all(ctxs.data(), gpus));
        a.shard_count = gpus;
        // NCCL sets its channels up on the first collective (~100 ms): do that here, as part of start-up, not of the frame
        CHECK(rt_group_start());
        for (int g = 0; g < gpus; g++) CHECK(rt_reduce(ctxs[(size_t)g], bufs[(size_t)g], 32, 0));
        CHECK(rt_group_end());
        for (int g = 0; g < gpus; g++) { ctx = ctxs[(size_t)g]; CHECK(rt_synchronize(ctx)); }
        ctx = ctxs[0];
    }

    // ---- render_init + render: what the reference's "took X seconds." brackets (main.cu:420-431) ----
    const auto t0 = std::chrono::steady_clock::now();
    if (gpus > 1) {
        std::vector<std::thread> th;
        std::vector<int> rcs(ctxs.size(), 0);
        std::vector<rt_render_stats> sts(ctxs.size());
        for (int g = 0; g < gpus; g++)
            th.emplace_back([&, g] {
                rt_render_args ag = a;
                ag.shard_rank = g;
                rcs[(size_t)g] = rt_render_accumulate(ctxs[(size_t)g], &ag, bufs[(size_t)g], &sts[(size_t)g]);
            });
        for (auto &t : th) t.join();
        for (int g = 0; g < gpus; g++) { ctx = ctxs[(size_t)g]; CHECK(rcs[(size_t)g]); st.rays += sts[(size_t)g].rays; st.kernel_ms = std::max(st.kernel_ms, sts[(size_t)g].kernel_ms); st.kernel_id = sts[(size_t)g].kernel_id; }
        ctx = ctxs[0];
        CHECK(rt_group_start());                          // the one exchange of the path: sum of the linear radiance buffers onto GPU 0
        for (int g = 0; g < gpus; g++) CHECK(rt_reduce(ctxs[(size_t)g], bufs[(size_t)g], n3, 0));
        CHECK(rt_group_end());
        CHECK(rt_finalize_ex(ctx, bufs[0], bufs[0], n3, ns, precision));     // /ns and sqrt on the sum (main.cu:111-114)
        CHECK(rt_synchronize(ctx));
    } else {
        CHECK(rt_render(ctx, &a, bufs[0], &st));
    }
    secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    std::cerr << "took " << secs << " seconds.\n";
    if (getenv("RT_VERBOSE"))
        std::cerr << "rays " << st.rays << ", kernel " << st.kernel_ms << " ms, " << (st.rays / (st.kernel_ms * 1e3)) << " Mrays/s on " << gpus
                  << " GPU(s), " << rt_kernel_name(st.kernel_id) << "\n";

    // ---- output switch (main.cu:435-453); the frame is quantised and formatted on the GPU, only the text crosses PCIe ----
    if (want_text) {
        CHECK(rt_ppm_format(ctx, bufs[0], nx, ny, &need));
        std::string txt(need, '\0');
        CHECK(rt_ppm_read(ctx, &txt[0], need));
        if (output_mode == 0) {
            std::cout.write(txt.data(), (std::streamsize)need);
        } else {
            std::ofstream out("output.ppm");
            out.write(txt.data(), (std::streamsize)need);
        }
    }
    for (size_t g = 0; g < ctxs.size(); g++) { rt_free(ctxs[g], bufs[g]); rt_destroy(ctxs[g]); }
    return 0;
}
