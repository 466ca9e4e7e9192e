/*
 * rt_oracle.h — CPU ORACLE (test infrastructure, NOT product code).
 *
 * A plain-C restatement of the render hot path of MuellerNico/DD2360-RayTracing
 * (reference file:line cited at every function in rt_oracle_core.inc.h).  Only
 * tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load this library; the product (librt_b200.so) never links or calls it.
 *
 * Parity pins (see DESIGN.md §3):
 *   - arithmetic mode RTO_ARITH_HOST (no FMA contraction) is checked bit-for-bit against
 *     oracle/_ref/ref_host_* — the reference's own headers compiled for the host — and
 *     against the fixtures under tests/golden/ref_host/ generated from it;
 *   - arithmetic mode RTO_ARITH_DEVICE (the FMA contraction pattern ptxas emits for the
 *     reference on sm_100, read from its SASS) is checked against frames produced by the
 *     reference's own kernels on a B200 (oracle/_ref/ref_cuda_*, fixtures under
 *     tests/golden/ref_cuda/).
 */
#ifndef RT_ORACLE_H
#define RT_ORACLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { RTO_MAT_NONE = -1, RTO_MAT_LAMBERTIAN = 0, RTO_MAT_METAL = 1, RTO_MAT_DIELECTRIC = 2 };
enum { RTO_ARITH_HOST = 0, RTO_ARITH_DEVICE = 1 };
/* per-pixel stream seeding: HEAD form main.cu:93, upstream form main.cu:90 (not restated: needs
 * cuRAND's skip-ahead matrices; rejected with an error) */
enum { RTO_SEED_HEAD = 0, RTO_SEED_UPSTREAM = 1 };

/* One sphere + its material, flattened (sphere.h:7-15, material.h:52-116). 36 bytes. */
typedef struct {
    float cx, cy, cz, radius;
    int32_t mat;          /* RTO_MAT_*; NONE = slot create_world never wrote (SURVEY D3) */
    float ax, ay, az;     /* albedo (lambertian, metal) */
    float param;          /* metal: fuzz (already clamped to <=1); dielectric: ref_idx */
} rto_sphere;

/* camera.h:51-58 */
typedef struct {
    float origin[3], lower_left_corner[3], horizontal[3], vertical[3], u[3], v[3], w[3];
    float lens_radius;
} rto_camera;

typedef struct {
    uint64_t rays;          /* closest-hit queries = iterations of the color() loop (main.cu:47) */
    uint64_t sphere_tests;  /* sphere::hit calls (sphere.h:17) */
    uint64_t aabb_tests;    /* intersect_ray_aabb calls (acceleration_structure.h:226) */
    uint64_t paths;         /* camera samples */
    uint32_t max_depth;
} rto_counters;

typedef struct {
    int32_t node_count, leaf_count;       /* Octree::nodeCount / leafCount (acceleration_structure.h:59-60) */
    int64_t entries;                      /* (cell, sphere) entries stored in leaves */
    int64_t dropped_full;                 /* "Leaf nodes full" drops (acceleration_structure.h:135) */
    int64_t dropped_outside;              /* "not in range of nodes AABB" drops (:105-108) */
} rto_octree_stats;

/* main.cu:146-181: fills out[0..n) (slots never written keep mat = NONE, zeros), returns #written. */
int rto_create_world(int n, float sphere_radius, rto_sphere *out);

/* main.cu:192-202 + camera.h:22-44.  arith picks how the constructor's float expressions round. */
void rto_camera_init(rto_camera *cam, int nx, int ny, int arith);

/* Byte size / layout of the reference's `Octree` for a given SPHERES_PER_LEAF
 * (acceleration_structure.h:23-61): nodes[585] (60 B), leaves[4097] (4*(spl+1) B), nodeCount, leafCount. */
size_t rto_octree_sizeof(int spl);
/* acceleration_structure.h:82-217, serial insertion.  blob must hold rto_octree_sizeof(spl) bytes. */
int rto_build_octree(const rto_sphere *spheres, int n, int spl, void *blob, rto_octree_stats *stats);

typedef struct {
    int nx, ny, ns;
    int use_octree;        /* USE_OCTREE (main.cu:24) */
    int spl;               /* SPHERES_PER_LEAF the blob was built with */
    int arith;             /* RTO_ARITH_* */
    int seed_mode;         /* RTO_SEED_* */
    int max_depth;         /* 50 (main.cu:47) */
    /* pixel subset: i in [i0,i1) step istep, j in [j0,j1) step jstep (full frame: 0,nx,1,0,ny,1) */
    int i0, i1, istep, j0, j1, jstep;
    int threads;           /* OpenMP threads, 0 = default */
} rto_render_params;

/* main.cu:96-117 (render) + :43-75 (color).  fb_gamma / fb_linear are nx*ny*3 floats (either may be NULL):
 * fb_gamma = what the reference stores in fb (after /ns and sqrt); fb_linear = the per-pixel sum before /ns.
 * Pixels outside the subset are left untouched. */
int rto_render(const rto_sphere *spheres, int n, const rto_camera *cam, const void *octree_blob,
               const rto_render_params *p, float *fb_gamma, float *fb_linear, rto_counters *ctr);

/* main.cu:321-333: P3 text exactly as output_to_stream writes it.  Returns bytes written (or needed if buf NULL). */
size_t rto_write_ppm(const float *fb_gamma, int nx, int ny, char *buf, size_t cap);
/* The same quantisation as bytes: out[(ny-1-j)*nx+i][c] = (uint8)int(255.99*fb). Row order = PPM order. */
void rto_quantise(const float *fb_gamma, int nx, int ny, uint8_t *out_rgb);

/* cuRAND XORWOW known-answer helper: first `count` outputs of curand() after curand_init(seed,0,0). */
void rto_xorwow_stream(uint64_t seed, int count, uint32_t *out_u32, float *out_uniform);
/* {d, v0..v4} after curand_init(seed, subsequence, 0): subsequence s starts 2^67 * s draws into the seed's stream. */
void rto_xorwow_state(uint64_t seed, uint64_t subsequence, uint32_t out6[6]);
/* the GF(2) skip matrices T^(2^(67+k)), k < max_bits (each 160 rows x 5 words); returns the number written */
int rto_xorwow_skip_tables(uint32_t *out, int max_bits);

/* Single-ray closest hit (for per-ray parity tests): returns sphere index or -1; t/normal out. */
int rto_closest_hit(const rto_sphere *spheres, int n, const void *octree_blob, int spl, int use_octree,
                    int arith, const float origin[3], const float dir[3], float *t_out);
/* rto_closest_hit for nrays rays (origins and directions: 3 floats each), OpenMP over the rays: out_idx[k], out_t[k]. */
void rto_closest_hits(const rto_sphere *spheres, int n, const void *octree_blob, int spl, int use_octree, int arith, int nrays,
                      const float *origins, const float *dirs, int *out_idx, float *out_t);

const char *rto_version(void);

#ifdef __cplusplus
}
#endif
#endif
