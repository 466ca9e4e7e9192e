/*
 * rt_oracle.c — CPU ORACLE (test infrastructure, NOT product code; see rt_oracle.h).
 *
 * Restates, in plain C, the render hot path of the reference (MuellerNico/DD2360-RayTracing):
 *   cuRAND XORWOW            /usr/local/cuda/include/curand_kernel.h:772-797,863-874 (CUDA 12.9, cuRAND 10.3.10;
 *                            third-party, not vendored by the reference), curand_uniform.h:69-72
 *   create_world             main.cu:146-204
 *   camera                   camera.h:22-49
 *   buildOctree / insert     acceleration_structure.h:82-217
 *   hitTree / traverseTree   acceleration_structure.h:226-342
 *   hitable_list / sphere    hitable_list.h:16-31, sphere.h:17-46
 *   materials                material.h:11-116
 *   render / color           main.cu:43-117
 *   PPM writer               main.cu:321-333
 * Build: gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC rt_oracle.c -lm   (see oracle/Makefile)
 */
#include "rt_oracle.h"

#include <float.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define RTO_TREE_HEIGHT 3       /* acceleration_structure.h:12 */
#define RTO_NUMBER_NODES 585    /* :13 */
#define RTO_NUMBER_LEAFS 4096   /* :14 */
#define RTO_NODE_INTS 15        /* OctNode = level + 6 floats + 8 children (:34-38) */

typedef struct { float x, y, z; } v3;
static inline v3 V3(float x, float y, float z) { v3 r = {x, y, z}; return r; }

/* ---- cuRAND XORWOW, subsequence 0 / offset 0 (no skip-ahead) ---- */
typedef struct { uint32_t d, v[5]; } xorwow;

static inline void xorwow_init(xorwow *s, uint64_t seed) {
    uint32_t s0 = (uint32_t)seed ^ 0xaad26b49u;
    uint32_t s1 = (uint32_t)(seed >> 32) ^ 0xf7dcefddu;
    uint32_t t0 = 1099087573u * s0;
    uint32_t t1 = 2591861531u * s1;
    s->d = 6615241u + t1 + t0;
    s->v[0] = 123456789u + t0;
    s->v[1] = 362436069u ^ t0;
    s->v[2] = 521288629u + t1;
    s->v[3] = 88675123u ^ t1;
    s->v[4] = 5783321u + t0;
}
static inline uint32_t xorwow_next(xorwow *s) {
    uint32_t t = s->v[0] ^ (s->v[0] >> 2);
    s->v[0] = s->v[1]; s->v[1] = s->v[2]; s->v[2] = s->v[3]; s->v[3] = s->v[4];
    s->v[4] = (s->v[4] ^ (s->v[4] << 4)) ^ (t ^ (t << 1));
    s->d += 362437u;
    return s->v[4] + s->d;
}
/* x * 2^-32 + 2^-33: the product is exact, so fused and unfused evaluation agree bit for bit */
static inline float xorwow_uniform(xorwow *s) {
    return (float)xorwow_next(s) * 2.3283064e-10f + (2.3283064e-10f / 2.0f);
}

/* ---- cuRAND XORWOW subsequences: curand_init(seed, subsequence, 0) (curand_kernel.h:772-797) --------------------------
 * Subsequence s starts 2^67 * s draws into the stream of the seed (XORWOW_SEQUENCE_SPACING 67, curand_precalc.h:54).
 * The five xorshift words advance LINEARLY over GF(2) (the Weyl counter d does not move: 362437 * 2^67 = 0 mod 2^32,
 * curand_kernel.h:697), so "skip 2^67 * s draws" is the 160x160 bit matrix T^(2^67 * s) applied to the words.  cuRAND
 * ships T^(2^67 * 4^k) as 218 KB of precalculated tables; this restatement derives them from the step function
 * itself: T by stepping the 160 unit vectors (as curand_kernel.h:569-586 does), S = T^(2^67) by 67 squarings, then
 * B[k] = S^(2^k), and applies B[k] for every set bit k of the subsequence number.  Powers of T commute, so this is
 * the same product cuRAND forms from its base-4 digits. */
#define RTO_SKIP_BITS 40
typedef struct { uint32_t row[160][5]; } gf2_mat;          /* row[i] = image of unit vector i (bit i%32 of word i/32) */
static gf2_mat g_skip[RTO_SKIP_BITS];
static int g_skip_ready = 0;

static void gf2_apply(const gf2_mat *m, const uint32_t in[5], uint32_t out[5]) {
    uint32_t r[5] = {0, 0, 0, 0, 0};
    for (int i = 0; i < 5; i++)
        for (int j = 0; j < 32; j++)
            if (in[i] >> j & 1u)
                for (int k = 0; k < 5; k++) r[k] ^= m->row[i * 32 + j][k];
    for (int k = 0; k < 5; k++) out[k] = r[k];
}
static void gf2_square(const gf2_mat *m, gf2_mat *out) {     /* out = m o m */
    gf2_mat t;
    for (int i = 0; i < 160; i++) gf2_apply(m, m->row[i], t.row[i]);
    *out = t;
}
static void skip_tables_init(void) {
#pragma omp critical(rto_skip_tables)
    if (!g_skip_ready) {
        gf2_mat t;
        for (int i = 0; i < 160; i++) {
            xorwow s;
            memset(&s, 0, sizeof s);
            s.v[i / 32] = 1u << (i & 31);
            xorwow_next(&s);
            for (int k = 0; k < 5; k++) t.row[i][k] = s.v[k];
        }
        for (int q = 0; q < 67; q++) gf2_square(&t, &t);
        g_skip[0] = t;
        for (int k = 1; k < RTO_SKIP_BITS; k++) gf2_square(&g_skip[k - 1], &g_skip[k]);
        g_skip_ready = 1;
    }
}
static void xorwow_init_subseq(xorwow *s, uint64_t seed, uint64_t subsequence) {
    xorwow_init(s, seed);
    if (!subsequence) return;
    if (!g_skip_ready) skip_tables_init();
    for (int k = 0; k < RTO_SKIP_BITS && subsequence >> k; k++)
        if (subsequence >> k & 1u) gf2_apply(&g_skip[k], s->v, s->v);
}
/* state words {d, v0..v4} after curand_init(seed, subsequence, 0) */
void rto_xorwow_state(uint64_t seed, uint64_t subsequence, uint32_t out6[6]) {
    xorwow s;
    xorwow_init_subseq(&s, seed, subsequence);
    out6[0] = s.d;
    for (int k = 0; k < 5; k++) out6[1 + k] = s.v[k];
}
/* the skip tables themselves (RTO_SKIP_BITS x 160 x 5 words), for checking the product's own copy */
int rto_xorwow_skip_tables(uint32_t *out, int max_bits) {
    if (!g_skip_ready) skip_tables_init();
    int nb = max_bits < RTO_SKIP_BITS ? max_bits : RTO_SKIP_BITS;
    if (out) memcpy(out, g_skip, (size_t)nb * sizeof(gf2_mat));
    return nb;
}

void rto_xorwow_stream(uint64_t seed, int count, uint32_t *out_u32, float *out_uniform) {
    xorwow a, b;
    xorwow_init(&a, seed);
    b = a;
    for (int i = 0; i < count; i++) {
        if (out_u32) out_u32[i] = xorwow_next(&a);
        if (out_uniform) out_uniform[i] = xorwow_uniform(&b);
    }
}

/* ---- scene: main.cu:146-181 ---- */
int rto_create_world(int n, float radius, rto_sphere *out) {
    xorwow rng;
    xorwow_init(&rng, 1984);                      /* rand_init, main.cu:80 */
    for (int k = 0; k < n; k++) {
        memset(&out[k], 0, sizeof out[k]);
        out[k].mat = RTO_MAT_NONE;
    }
    if (n < 4) return 0;
#define RND xorwow_uniform(&rng)
    out[0] = (rto_sphere){0.0f, -1000.0f, -1.0f, 1000.0f, RTO_MAT_LAMBERTIAN, 0.5f, 0.5f, 0.5f, 0.0f};
    int i = 1;
    out[i++] = (rto_sphere){0.0f, 1.0f, 0.0f, 1.0f, RTO_MAT_DIELECTRIC, 0, 0, 0, 1.5f};
    out[i++] = (rto_sphere){-4.0f, 1.0f, 0.0f, 1.0f, RTO_MAT_LAMBERTIAN, 0.4f, 0.2f, 0.1f, 0.0f};
    out[i++] = (rto_sphere){4.0f, 1.0f, 0.0f, 1.0f, RTO_MAT_METAL, 0.7f, 0.6f, 0.5f, 0.0f};
    const int spheres_per_dim = (int)sqrtf((float)n - 4);          /* main.cu:160 */
    const double spacing = 20. / spheres_per_dim;                  /* :161 */
    for (double a = -10; a < 10; a += spacing) {
        for (double b = -10; b < 10 && i < n; b += spacing) {
            const float choose_mat = RND;
            /* device order of evaluation is left to right (SURVEY D4) */
            const float cx = (float)(a + RND);
            const float cz = (float)(b + RND);
            rto_sphere s = {cx, radius, cz, radius, 0, 0, 0, 0, 0};
            if (choose_mat < 0.8f) {
                s.mat = RTO_MAT_LAMBERTIAN;
                float r0 = RND, r1 = RND, r2 = RND, r3 = RND, r4 = RND, r5 = RND;
                s.ax = r0 * r1; s.ay = r2 * r3; s.az = r4 * r5;
            } else if (choose_mat < 0.95f) {
                s.mat = RTO_MAT_METAL;
                float r0 = RND, r1 = RND, r2 = RND, r3 = RND;
                s.ax = 0.5f * (1.0f + r0); s.ay = 0.5f * (1.0f + r1); s.az = 0.5f * (1.0f + r2);
                float f = 0.5f * r3;
                s.param = f < 1.0f ? f : 1.0f;                     /* material.h:67 */
            } else {
                s.mat = RTO_MAT_DIELECTRIC;
                s.param = 1.5f;
            }
            out[i++] = s;
        }
    }
#undef RND
    return i;
}

/* ---- camera: main.cu:192-202, camera.h:22-44 ---- */
static v3 cross3(v3 a, v3 b, int fma) {
    /* vec3.h:95-99; device: a*b - c*d -> fma(a,b,-(c*d)) */
    if (fma)
        return V3(fmaf(a.y, b.z, -(a.z * b.y)), -fmaf(a.x, b.z, -(a.z * b.x)), fmaf(a.x, b.y, -(a.y * b.x)));
    return V3(a.y * b.z - a.z * b.y, -(a.x * b.z - a.z * b.x), a.x * b.y - a.y * b.x);
}
static v3 unit3(v3 v, int fma) {
    float l2 = fma ? fmaf(v.z, v.z, fmaf(v.x, v.x, v.y * v.y)) : (v.x * v.x + v.y * v.y) + v.z * v.z;
    float l = sqrtf(l2);
    return V3(v.x / l, v.y / l, v.z / l);
}
void rto_camera_init(rto_camera *c, int nx, int ny, int arith) {
    /* lookfrom, lookat, vup, vfov, aperture and focus distance are compile-time constants in the reference:
     * nvcc folds w, u, v, half_height with separate roundings (LLVM constant folding happens before FMA
     * contraction), so only the aspect-dependent products can be fused on the device. */
    const v3 lookfrom = V3(13, 2, 3), lookat = V3(0, 0, 0), vup = V3(0, 1, 0);
    const float vfov = 30.0f, aperture = 0.1f, focus = 10.0f;
    const float aspect = (float)nx / (float)ny;
    c->lens_radius = aperture / 2.0f;
    float theta = vfov * ((float)M_PI) / 180.0f;
    float arg = theta / 2.0f;
    float half_height = tanf(arg);
    float half_width = aspect * half_height;
    v3 w = unit3(V3(lookfrom.x - lookat.x, lookfrom.y - lookat.y, lookfrom.z - lookat.z), 0);
    v3 u = unit3(cross3(vup, w, 0), 0);
    v3 v = cross3(w, u, 0);
    float hw = half_width * focus, hh = half_height * focus;
    float O[3] = {lookfrom.x, lookfrom.y, lookfrom.z};
    float U[3] = {u.x, u.y, u.z}, Vv[3] = {v.x, v.y, v.z}, W[3] = {w.x, w.y, w.z};
    for (int k = 0; k < 3; k++) {
        c->origin[k] = O[k];
        c->u[k] = U[k]; c->v[k] = Vv[k]; c->w[k] = W[k];
        if (arith == RTO_ARITH_DEVICE) {
            /* origin - hw*u - hh*v - focus*w: the first two products are fused into the subtraction; focus*w
             * is a compile-time constant in the reference (folded, so rounded on its own) */
            float t = fmaf(-hw, U[k], O[k]);
            t = fmaf(-hh, Vv[k], t);
            c->lower_left_corner[k] = t - focus * W[k];
        } else {
            c->lower_left_corner[k] = ((O[k] - hw * U[k]) - hh * Vv[k]) - focus * W[k];
        }
        c->horizontal[k] = (2.0f * half_width * focus) * U[k];
        c->vertical[k] = (2.0f * half_height * focus) * Vv[k];
    }
}

/* ---- octree blob (acceleration_structure.h:23-61) ---- */
typedef struct {
    int32_t *nodes;      /* 585 * 15 ints */
    int32_t *leaves;     /* 4097 * (spl+1) ints */
    int32_t *counts;     /* nodeCount, leafCount */
    int spl, leaf_count;
} oct_view;

size_t rto_octree_sizeof(int spl) {
    return (size_t)RTO_NUMBER_NODES * RTO_NODE_INTS * 4 + (size_t)(RTO_NUMBER_LEAFS + 1) * (size_t)(spl + 1) * 4 + 8;
}
static oct_view oct_open(void *blob, int spl) {
    oct_view v;
    v.nodes = (int32_t *)blob;
    v.leaves = v.nodes + RTO_NUMBER_NODES * RTO_NODE_INTS;
    v.counts = v.leaves + (size_t)(RTO_NUMBER_LEAFS + 1) * (size_t)(spl + 1);
    v.spl = spl;
    v.leaf_count = v.counts[1];
    return v;
}
static inline int32_t *oct_node(const oct_view *v, int i) { return v->nodes + (size_t)i * RTO_NODE_INTS; }
static inline int32_t *oct_leaf(const oct_view *v, int i) { return v->leaves + (size_t)i * (size_t)(v->spl + 1); }

/* acceleration_structure.h:82-93: x uses (low, high], y and z use [low, high] */
static int sphere_in_box(const rto_sphere *s, const float *bx) {
    float xl = bx[0] - s->radius, yl = bx[1] - s->radius, zl = bx[2] - s->radius;
    float xh = bx[3] + s->radius, yh = bx[4] + s->radius, zh = bx[5] + s->radius;
    return (s->cx > xl && s->cx <= xh) && (s->cy >= yl && s->cy <= yh) && (s->cz >= zl && s->cz <= zh);
}

/* acceleration_structure.h:104-186 */
static int oct_insert(oct_view *ov, int node, const rto_sphere *s, int idx, rto_octree_stats *st) {
    int32_t *nd = oct_node(ov, node);
    const float *bx = (const float *)(nd + 1);
    int32_t *children = nd + 7;
    if (!sphere_in_box(s, bx)) { st->dropped_outside++; return 0; }
    if (nd[0] == RTO_TREE_HEIGHT) {
        for (int i = 0; i < 8; i++) {
            int leaf = children[i];
            if (leaf == 0) {
                leaf = ov->counts[1]++;
                memset(oct_leaf(ov, leaf), 0, (size_t)(ov->spl + 1) * 4);
                children[i] = leaf;
            }
            int32_t *lf = oct_leaf(ov, leaf);
            if (lf[ov->spl] < ov->spl) { lf[lf[ov->spl]++] = idx; st->entries++; return 1; }
        }
        st->dropped_full++;
        return 0;
    }
    int inserted = 0;
    float xl = bx[0], yl = bx[1], zl = bx[2], xh = bx[3], yh = bx[4], zh = bx[5];
    float xm = xl + (xh - xl) / 2, ym = yl + (yh - yl) / 2, zm = zl + (zh - zl) / 2;   /* :141-147 */
    const float cb[8][6] = {                                                           /* :150-165 */
        {xl, yl, zl, xm, ym, zm}, {xl, yl, zm, xm, ym, zh}, {xl, ym, zl, xm, yh, zm}, {xl, ym, zm, xm, yh, zh},
        {xm, yl, zl, xh, ym, zm}, {xm, yl, zm, xh, ym, zh}, {xm, ym, zl, xh, yh, zm}, {xm, ym, zm, xh, yh, zh}};
    for (int i = 0; i < 8; i++) {
        if (sphere_in_box(s, cb[i])) {
            if (children[i] == 0) {
                int nn = ov->counts[0]++;
                children[i] = nn;
                int32_t *c = oct_node(ov, nn);
                memset(c, 0, RTO_NODE_INTS * 4);
                c[0] = nd[0] + 1;
                memcpy(c + 1, cb[i], 24);
            }
            inserted += oct_insert(ov, children[i], s, idx, st);
        }
    }
    return inserted;
}

/* acceleration_structure.h:195-217 */
int rto_build_octree(const rto_sphere *sph, int n, int spl, void *blob, rto_octree_stats *stats) {
    rto_octree_stats st;
    memset(&st, 0, sizeof st);
    memset(blob, 0, rto_octree_sizeof(spl));          /* `new Octree()` value-initialises */
    oct_view ov = oct_open(blob, spl);
    ov.counts[0] = 0; ov.counts[1] = 1;               /* nodeCount = 0, leafCount = 1 (:59-60) */
    int32_t *root = oct_node(&ov, 0);
    const float rb[6] = {-11, 0, -11, 11, 2, 11};     /* :203 */
    root[0] = 0;
    memcpy(root + 1, rb, 24);
    ov.counts[0]++;
    for (int i = 1; i < n; i++) oct_insert(&ov, 0, &sph[i], i, &st);   /* ground (idx 0) skipped, :208 */
    st.node_count = ov.counts[0];
    st.leaf_count = ov.counts[1];
    if (stats) *stats = st;
    return 0;
}

/* ---- the two arithmetic instantiations ---- */
#define RTO_FMA 0
#include "rt_oracle_core.inc.h"
#undef RTO_FMA
#define RTO_FMA 1
#include "rt_oracle_core.inc.h"
#undef RTO_FMA

int rto_render(const rto_sphere *sph, int n, const rto_camera *cam, const void *blob, const rto_render_params *p,
               float *fb_gamma, float *fb_linear, rto_counters *ctr_out) {
    if (p->seed_mode != RTO_SEED_HEAD && p->seed_mode != RTO_SEED_UPSTREAM) return -2;
    if (p->seed_mode == RTO_SEED_UPSTREAM && !g_skip_ready) skip_tables_init();
    if (p->use_octree && !blob) return -1;
    oct_view ov;
    memset(&ov, 0, sizeof ov);
    if (p->use_octree) ov = oct_open((void *)blob, p->spl);
    rto_counters total;
    memset(&total, 0, sizeof total);
    int nrows = (p->j1 - p->j0 + p->jstep - 1) / p->jstep;
#ifdef _OPENMP
    if (p->threads > 0) omp_set_num_threads(p->threads);
#endif
#pragma omp parallel
    {
        rto_counters c;
        memset(&c, 0, sizeof c);
#pragma omp for schedule(dynamic, 1)
        for (int r = 0; r < nrows; r++) {
            int j = p->j0 + r * p->jstep;
            for (int i = p->i0; i < p->i1; i += p->istep) {
                if (p->arith == RTO_ARITH_DEVICE) render_pixel_dev(sph, n, cam, &ov, p, i, j, fb_gamma, fb_linear, &c);
                else render_pixel_host(sph, n, cam, &ov, p, i, j, fb_gamma, fb_linear, &c);
            }
        }
#pragma omp critical
        {
            total.rays += c.rays; total.sphere_tests += c.sphere_tests; total.aabb_tests += c.aabb_tests;
            total.paths += c.paths;
            if (c.max_depth > total.max_depth) total.max_depth = c.max_depth;
        }
    }
    if (ctr_out) *ctr_out = total;
    return 0;
}

int rto_closest_hit(const rto_sphere *sph, int n, const void *blob, int spl, int use_octree, int arith,
                    const float o[3], const float d[3], float *t_out) {
    oct_view ov;
    memset(&ov, 0, sizeof ov);
    if (use_octree) ov = oct_open((void *)blob, spl);
    v3 O = V3(o[0], o[1], o[2]), D = V3(d[0], d[1], d[2]);
    return arith == RTO_ARITH_DEVICE ? closest_hit_dev(sph, n, &ov, use_octree, O, D, t_out)
                                     : closest_hit_host(sph, n, &ov, use_octree, O, D, t_out);
}

void rto_closest_hits(const rto_sphere *sph, int n, const void *blob, int spl, int use_octree, int arith, int nrays,
                      const float *org, const float *dir, int *out_idx, float *out_t) {
#pragma omp parallel for schedule(dynamic, 64)
    for (int k = 0; k < nrays; k++)
        out_idx[k] = rto_closest_hit(sph, n, blob, spl, use_octree, arith, org + 3 * (size_t)k, dir + 3 * (size_t)k, out_t + k);
}

/* main.cu:321-333 */
void rto_quantise(const float *fb, int nx, int ny, uint8_t *out) {
    for (int j = ny - 1; j >= 0; j--)
        for (int i = 0; i < nx; i++) {
            size_t pi = (size_t)j * nx + i, po = (size_t)(ny - 1 - j) * nx + i;
            for (int c = 0; c < 3; c++) out[3 * po + c] = (uint8_t)(int)(255.99 * fb[3 * pi + c]);
        }
}
size_t rto_write_ppm(const float *fb, int nx, int ny, char *buf, size_t cap) {
    size_t off = 0;
    char line[64];
    int k = snprintf(line, sizeof line, "P3\n%d %d\n255\n", nx, ny);
    if (buf && off + (size_t)k <= cap) memcpy(buf + off, line, (size_t)k);
    off += (size_t)k;
    for (int j = ny - 1; j >= 0; j--)
        for (int i = 0; i < nx; i++) {
            size_t pi = (size_t)j * nx + i;
            int ir = (int)(255.99 * fb[3 * pi + 0]), ig = (int)(255.99 * fb[3 * pi + 1]), ib = (int)(255.99 * fb[3 * pi + 2]);
            k = snprintf(line, sizeof line, "%d %d %d\n", ir, ig, ib);
            if (buf && off + (size_t)k <= cap) memcpy(buf + off, line, (size_t)k);
            off += (size_t)k;
        }
    return off;
}

const char *rto_version(void) { return "rt_oracle 1 (restates MuellerNico/DD2360-RayTracing render path)"; }
