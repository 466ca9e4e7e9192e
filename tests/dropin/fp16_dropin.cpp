// Test program for the device-side members of include/rt_dropin.h compiled with -DUSE_FP16 (needs a GPU): buildOctree returns
// the USE_FP16 Octree layout, hitTree / material::scatter / camera::get_ray answer as the reference's FP16 build does.
//   stdin : n, then n lines "cx cy cz r mat ax ay az param" (hex floats); q, then q lines "ox oy oz dx dy dz"; g, then g lines "s t seed"
//   stdout: "octree nodeCount leafCount sizeof(Octree) digest", one line per query ray
//           ("idx t px py pz nx ny nz scattered sox soy soz ax ay az dx dy dz next_draw" or "-1"), one line per get_ray
#include <cstdio>
#include <vector>

#include "rt_dropin.h"

#ifndef USE_FP16
#error "build with -DUSE_FP16"
#endif

int main() {
    int n = 0;
    if (scanf("%d", &n) != 1) return 1;
    std::vector<sphere> spheres((size_t)n);
    std::vector<hitable *> list;
    for (int i = 0; i < n; i++) {
        float cx, cy, cz, r, ax, ay, az, p;
        int mat;
        if (scanf("%a %a %a %a %d %a %a %a %a", &cx, &cy, &cz, &r, &mat, &ax, &ay, &az, &p) != 9) return 2;
        material *m = nullptr;
        if (mat == RT_MAT_LAMBERTIAN) m = new lambertian(vec3(ax, ay, az));
        else if (mat == RT_MAT_METAL) m = new metal(vec3(ax, ay, az), p);
        else if (mat == RT_MAT_DIELECTRIC) m = new dielectric(p);
        spheres[(size_t)i] = sphere(vec3(cx, cy, cz), r, m);
    }
    for (int i = 0; i < n; i++) list.push_back(&spheres[(size_t)i]);
    hitable *world = new hitable_list(list.data(), n);

    rt_context *ctx = nullptr;
    if (rt_create(0, &ctx)) { fprintf(stderr, "rt_create failed\n"); return 3; }
    rt_dropin_bind(ctx);
    Octree *octree = buildOctree(spheres.data(), n);                 // acceleration_structure.h:195
    if (!octree) { fprintf(stderr, "buildOctree: %s\n", rt_last_error(ctx)); return 4; }
    unsigned long long h = 1469598103934665603ull;                  // FNV-1a over the blob
    const unsigned char *b = reinterpret_cast<const unsigned char *>(octree);
    for (size_t i = 0; i < sizeof(Octree); i++) { h ^= b[i]; h *= 1099511628211ull; }
    printf("octree %d %d %zu %016llx\n", octree->nodeCount, octree->leafCount, sizeof(Octree), h);

    int q = 0;
    if (scanf("%d", &q) != 1) return 5;
    for (int k = 0; k < q; k++) {
        float ox, oy, oz, dx, dy, dz;
        if (scanf("%a %a %a %a %a %a", &ox, &oy, &oz, &dx, &dy, &dz) != 6) return 6;
        const ray r(vec3(ox, oy, oz), vec3(dx, dy, dz));
        hit_record rec;
        if (!hitTree(octree, r, rec, &world)) { printf("-1\n"); continue; }         // acceleration_structure.h:319
        curandState st;
        curand_init(1984 + k, 0, 0, &st);
        vec3 att;
        ray sc;
        const bool go = rec.mat_ptr->scatter(r, rec, att, sc, &st);                   // material.h:55,68,81
        printf("%d %a %a %a %a %a %a %a %d %a %a %a %a %a %a %a %a %a %u\n", rec.sphere_index, rec.t, rec.p.x(), rec.p.y(), rec.p.z(),
               rec.normal.x(), rec.normal.y(), rec.normal.z(), go ? 1 : 0, sc.origin().x(), sc.origin().y(), sc.origin().z(), att.x(),
               att.y(), att.z(), sc.direction().x(), sc.direction().y(), sc.direction().z(), curand(&st));
    }
    int g = 0;
    if (scanf("%d", &g) != 1) return 7;
    camera cam(vec3(13, 2, 3), vec3(0, 0, 0), vec3(0, 1, 0), 30.0f, 1.5f, 0.1f, 10.0f);     // main.cu:192-202 at 1200x800
    if (rt_apply_camera(ctx, cam, 1200, 800)) return 8;
    for (int k = 0; k < g; k++) {
        float s, t;
        unsigned long long seed;
        if (scanf("%a %a %llu", &s, &t, &seed) != 3) return 9;
        curandState st;
        curand_init(seed, 0, 0, &st);
        const ray r = cam.get_ray(s, t, &st);                                          // camera.h:45
        printf("%a %a %a %a %a %a %u\n", r.origin().x(), r.origin().y(), r.origin().z(), r.direction().x(), r.direction().y(), r.direction().z(),
               curand(&st));
    }
    delete octree;
    rt_destroy(ctx);
    return 0;
}
