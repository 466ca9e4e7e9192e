/*
 * rt_dropin.h — the reference's world-building class surface, host side, over the C ABI of rt_abi.h.
 *
 * In the reference these classes live on the device: create_world (main.cu:146-204) news up `sphere`, `lambertian`,
 * `metal`, `dielectric`, a `hitable_list` and a `camera` inside a one-thread kernel, and render chases their vtables.
 * Code written against that surface keeps compiling against this header — same class names, constructor signatures
 * and accessors (vec3.h, ray.h, hitable.h:11-21, sphere.h:7-15, hitable_list.h:6-14, material.h:47-116,
 * camera.h:20-58) — but the objects are plain host descriptions: `rt_upload_world` flattens a `hitable` tree into the
 * SoA scene of librt_b200.so (rt_scene_upload) and `rt_apply_camera` hands the constructor arguments to
 * rt_camera_set.  Nothing here runs on the GPU; the rendering arithmetic is the library's.
 *
 * `hitable::hit` is provided for host-side picking / debugging with the reference's semantics (closest hit, strict
 * '<'); it is NOT the render path.
 *
 * The device-side members of the reference surface — `camera::get_ray` (camera.h:45), `material::scatter`
 * (material.h:55-113), `buildOctree` (acceleration_structure.h:195) and `hitTree` (:319) — are here too, with the
 * reference's signatures; they forward to the library (rt_camera_get_rays, rt_scatter_rays, rt_octree_build +
 * rt_octree_export_reference, rt_trace_rays), so the arithmetic is the GPU's and the results are the ones the render
 * kernels compute.  The context they talk to is the one bound with rt_dropin_bind().  `curandState` is the XORWOW state
 * {d, v[5]} and `curand_init` / `curand_uniform` follow cuRAND (subsequence < 2^40, offset 0).
 *
 * Compiled with -DUSE_FP16 (the reference's precision switch, precision_types.h:8) those members answer as the reference's
 * USE_FP16 build does: hitTree, camera::get_ray and material::scatter forward with RT_PREC_FP16 (rt_trace_rays_ex,
 * rt_camera_get_rays_ex, rt_scatter_rays_ex), buildOctree builds with rt_octree_build_ex(.., RT_PREC_FP16, ..) and returns
 * that build's layout (AABB of six halves, 48-byte nodes), and hitTree's rec.t, rec.p and rec.normal are the half values the
 * library computes.  The host real_t stays float: every value crossing into the library is rounded to half there, every
 * value coming back is a half widened to float (so it goes back in exactly), and arithmetic the caller does between member
 * calls is the caller's own, in float — it is not the reference's half arithmetic.
 */
#ifndef RT_DROPIN_H
#define RT_DROPIN_H

#include <float.h>
#include <math.h>
#include <string.h>

#include <vector>

#include "rt_abi.h"

/* the context the device-side members of this surface forward to */
inline rt_context *&rt_dropin_context() { static rt_context *ctx = nullptr; return ctx; }
inline void rt_dropin_bind(rt_context *ctx) { rt_dropin_context() = ctx; }

/* curand_kernel.h:772-797 / curand_uniform.h:69-72, host side: the stream a pixel draws from (main.cu:84-94) */
struct curandState { uint32_t d, v[5]; };
inline void curand_init(unsigned long long seed, unsigned long long subsequence, unsigned long long /*offset: 0*/, curandState *st) {
    uint32_t w[6];
    rt_xorwow_state(seed, subsequence, w);
    st->d = w[0];
    for (int k = 0; k < 5; k++) st->v[k] = w[1 + k];
}
inline uint32_t curand(curandState *s) {
    const uint32_t t = s->v[0] ^ (s->v[0] >> 2);
    s->v[0] = s->v[1]; s->v[1] = s->v[2]; s->v[2] = s->v[3]; s->v[3] = s->v[4];
    s->v[4] = (s->v[4] ^ (s->v[4] << 4)) ^ (t ^ (t << 1));
    s->d += 362437u;
    return s->v[4] + s->d;
}
inline float curand_uniform(curandState *s) { return fmaf((float)curand(s), 2.3283064e-10f, 1.16415321826934814453125e-10f); }

typedef float real_t;                                   /* precision_types.h:179; USE_FP16 is a run-time switch of the library */

class vec3 {
public:
    vec3() { e[0] = e[1] = e[2] = 0; }
    vec3(real_t e0, real_t e1, real_t e2) { e[0] = e0; e[1] = e1; e[2] = e2; }
    real_t x() const { return e[0]; }
    real_t y() const { return e[1]; }
    real_t z() const { return e[2]; }
    real_t r() const { return e[0]; }
    real_t g() const { return e[1]; }
    real_t b() const { return e[2]; }
    const vec3 &operator+() const { return *this; }
    vec3 operator-() const { return vec3(-e[0], -e[1], -e[2]); }
    real_t operator[](int i) const { return e[i]; }
    real_t &operator[](int i) { return e[i]; }
    vec3 &operator+=(const vec3 &v) { for (int i = 0; i < 3; i++) e[i] += v.e[i]; return *this; }
    vec3 &operator-=(const vec3 &v) { for (int i = 0; i < 3; i++) e[i] -= v.e[i]; return *this; }
    vec3 &operator*=(const vec3 &v) { for (int i = 0; i < 3; i++) e[i] *= v.e[i]; return *this; }
    vec3 &operator/=(const vec3 &v) { for (int i = 0; i < 3; i++) e[i] /= v.e[i]; return *this; }
    vec3 &operator*=(real_t t) { for (int i = 0; i < 3; i++) e[i] *= t; return *this; }
    vec3 &operator/=(real_t t) { const real_t k = (real_t)(1.0 / t); for (int i = 0; i < 3; i++) e[i] *= k; return *this; }
    real_t squared_length() const { return e[0] * e[0] + e[1] * e[1] + e[2] * e[2]; }
    real_t length() const { return sqrtf(squared_length()); }
    void make_unit_vector() { *this /= length(); }
    real_t e[3];
};
inline vec3 operator+(const vec3 &a, const vec3 &b) { return vec3(a.e[0] + b.e[0], a.e[1] + b.e[1], a.e[2] + b.e[2]); }
inline vec3 operator-(const vec3 &a, const vec3 &b) { return vec3(a.e[0] - b.e[0], a.e[1] - b.e[1], a.e[2] - b.e[2]); }
inline vec3 operator*(const vec3 &a, const vec3 &b) { return vec3(a.e[0] * b.e[0], a.e[1] * b.e[1], a.e[2] * b.e[2]); }
inline vec3 operator/(const vec3 &a, const vec3 &b) { return vec3(a.e[0] / b.e[0], a.e[1] / b.e[1], a.e[2] / b.e[2]); }
inline vec3 operator*(real_t t, const vec3 &v) { return vec3(t * v.e[0], t * v.e[1], t * v.e[2]); }
inline vec3 operator*(const vec3 &v, real_t t) { return t * v; }
inline vec3 operator/(const vec3 &v, real_t t) { return vec3(v.e[0] / t, v.e[1] / t, v.e[2] / t); }
inline real_t dot(const vec3 &a, const vec3 &b) { return a.e[0] * b.e[0] + a.e[1] * b.e[1] + a.e[2] * b.e[2]; }
inline vec3 cross(const vec3 &a, const vec3 &b) {
    return vec3(a.e[1] * b.e[2] - a.e[2] * b.e[1], -(a.e[0] * b.e[2] - a.e[2] * b.e[0]), a.e[0] * b.e[1] - a.e[1] * b.e[0]);
}
inline vec3 unit_vector(const vec3 &v) { return v / v.length(); }

class ray {
public:
    ray() {}
    ray(const vec3 &a, const vec3 &b) : A(a), B(b) {}
    vec3 origin() const { return A; }
    vec3 direction() const { return B; }
    vec3 point_at_parameter(real_t t) const { return A + t * B; }
    vec3 A, B;
};

/* ---- materials (material.h:47-116): descriptions only ------------------------------------------------------------------ */
struct hit_record;
class material {
public:
    virtual ~material() {}
    virtual void describe(rt_sphere_desc &d) const = 0;      /* fills mat, albedo, param */
    /* material.h:55,68,81 — evaluated by the library for the sphere the record came from (rec.sphere_index in the bound
     * context's scene, set by hitTree / rt_hit_list below); false = absorbed */
    inline bool scatter(const ray &r_in, const hit_record &rec, vec3 &attenuation, ray &scattered, curandState *local_rand_state) const;
};
class lambertian : public material {
public:
    explicit lambertian(const vec3 &a) : albedo(a) {}
    void describe(rt_sphere_desc &d) const override { d.mat = RT_MAT_LAMBERTIAN; d.ax = albedo.x(); d.ay = albedo.y(); d.az = albedo.z(); d.param = 0; }
    vec3 albedo;
};
class metal : public material {
public:
    metal(const vec3 &a, real_t f) : albedo(a), fuzz(f < 1.0f ? f : 1.0f) {}       /* the clamp of material.h:66 */
    void describe(rt_sphere_desc &d) const override { d.mat = RT_MAT_METAL; d.ax = albedo.x(); d.ay = albedo.y(); d.az = albedo.z(); d.param = fuzz; }
    vec3 albedo;
    real_t fuzz;
};
class dielectric : public material {
public:
    explicit dielectric(real_t ri) : ref_idx(ri) {}
    void describe(rt_sphere_desc &d) const override { d.mat = RT_MAT_DIELECTRIC; d.ax = d.ay = d.az = 0; d.param = ref_idx; }
    real_t ref_idx;
};

/* ---- geometry (hitable.h, sphere.h, hitable_list.h) --------------------------------------------------------------------- */
struct hit_record {
    real_t t;
    vec3 p;
    vec3 normal;
    material *mat_ptr;
    int sphere_index = -1;      /* extension: index of the hit sphere in the uploaded world (what mat_ptr identifies in the reference) */
};
inline bool material::scatter(const ray &r_in, const hit_record &rec, vec3 &attenuation, ray &scattered, curandState *st) const {
    rt_context *ctx = rt_dropin_context();
    if (!ctx || rec.sphere_index < 0) return false;
    const float o[3] = {r_in.A[0], r_in.A[1], r_in.A[2]}, d[3] = {r_in.B[0], r_in.B[1], r_in.B[2]};
    uint32_t w[6] = {st->d, st->v[0], st->v[1], st->v[2], st->v[3], st->v[4]};
    float p[3], nrm[3], od[3], att[3];
    int go = 0;
#ifdef USE_FP16
    if (rt_scatter_rays_ex(ctx, RT_PREC_FP16, 1, &rec.sphere_index, o, d, &rec.t, w, p, nrm, od, att, &go) != 0 || go < 0) return false;
#else
    if (rt_scatter_rays(ctx, 1, &rec.sphere_index, o, d, &rec.t, w, p, nrm, od, att, &go) != 0 || go < 0) return false;
#endif
    st->d = w[0];
    for (int k = 0; k < 5; k++) st->v[k] = w[1 + k];
    attenuation = vec3(att[0], att[1], att[2]);
    scattered = ray(vec3(p[0], p[1], p[2]), vec3(od[0], od[1], od[2]));
    return go == 1;
}
class hitable {
public:
    virtual ~hitable() {}
    virtual bool hit(const ray &r, real_t t_min, real_t t_max, hit_record &rec) const = 0;
    virtual void flatten(std::vector<rt_sphere_desc> &out) const = 0;     /* appends this object's spheres, in list order */
};
class sphere : public hitable {
public:
    sphere() : radius(0), mat_ptr(nullptr) {}
    sphere(vec3 cen, real_t r, material *m) : center(cen), radius(r), mat_ptr(m) {}
    bool hit(const ray &r, real_t t_min, real_t t_max, hit_record &rec) const override {
        const vec3 oc = r.origin() - center;
        const real_t a = dot(r.direction(), r.direction()), b = dot(oc, r.direction()), c = dot(oc, oc) - radius * radius;
        const real_t disc = b * b - a * c;
        if (!(disc > 0)) return false;
        const real_t sq = sqrtf(disc);
        for (int k = 0; k < 2; k++) {
            const real_t t = (k == 0 ? (-b - sq) : (-b + sq)) / a;
            if (t < t_max && t > t_min) {
                rec.t = t;
                rec.p = r.point_at_parameter(t);
                rec.normal = (rec.p - center) / radius;
                rec.mat_ptr = mat_ptr;
                return true;
            }
        }
        return false;
    }
    void flatten(std::vector<rt_sphere_desc> &out) const override {
        rt_sphere_desc d;
        d.cx = center.x(); d.cy = center.y(); d.cz = center.z(); d.radius = radius;
        d.mat = RT_MAT_NONE; d.ax = d.ay = d.az = d.param = 0;
        if (mat_ptr) mat_ptr->describe(d);
        out.push_back(d);
    }
    vec3 center;
    real_t radius;
    material *mat_ptr;
};
class hitable_list : public hitable {
public:
    hitable_list() : list(nullptr), list_size(0) {}
    hitable_list(hitable **l, int n) : list(l), list_size(n) {}
    bool hit(const ray &r, real_t t_min, real_t t_max, hit_record &rec) const override {
        hit_record tmp;
        bool any = false;
        real_t closest = t_max;
        for (int i = 0; i < list_size; i++)
            if (list[i]->hit(r, t_min, closest, tmp)) { any = true; closest = tmp.t; rec = tmp; }
        return any;
    }
    void flatten(std::vector<rt_sphere_desc> &out) const override { for (int i = 0; i < list_size; i++) list[i]->flatten(out); }
    hitable **list;
    int list_size;
};

/* ---- camera (camera.h:20-58): keeps the constructor's arguments ------------------------------------------------------------ */
class camera {
public:
    camera(vec3 lookfrom, vec3 lookat, vec3 vup, real_t vfov, real_t aspect, real_t aperture, real_t focus_dist) {
        for (int k = 0; k < 3; k++) { desc.lookfrom[k] = lookfrom[k]; desc.lookat[k] = lookat[k]; desc.vup[k] = vup[k]; }
        desc.vfov = vfov; desc.aspect = aspect; desc.aperture = aperture; desc.focus_dist = focus_dist;
    }
    /* camera.h:45-49, evaluated by the library with the camera of the bound context (rt_apply_camera first) */
    ray get_ray(real_t s, real_t t, curandState *local_rand_state) const {
        rt_context *ctx = rt_dropin_context();
        uint32_t w[6] = {local_rand_state->d, local_rand_state->v[0], local_rand_state->v[1], local_rand_state->v[2], local_rand_state->v[3],
                         local_rand_state->v[4]};
        float o[3] = {0, 0, 0}, d[3] = {0, 0, 0};
#ifdef USE_FP16
        if (ctx && rt_camera_get_rays_ex(ctx, RT_PREC_FP16, 1, &s, &t, w, o, d) == 0) {
#else
        if (ctx && rt_camera_get_rays(ctx, 1, &s, &t, w, o, d) == 0) {
#endif
            local_rand_state->d = w[0];
            for (int k = 0; k < 5; k++) local_rand_state->v[k] = w[1 + k];
        }
        return ray(vec3(o[0], o[1], o[2]), vec3(d[0], d[1], d[2]));
    }
    rt_camera_desc desc;
};

/* the world a `hitable*` describes -> the library's scene; index 0 of the flattened list is the sphere hitTree tests
 * unconditionally (the "ground" of acceleration_structure.h:322), as in the reference's d_list */
inline int rt_upload_world(rt_context *ctx, const hitable *world) {
    std::vector<rt_sphere_desc> flat;
    world->flatten(flat);
    return rt_scene_upload(ctx, flat.data(), (int)flat.size());
}
inline int rt_apply_camera(rt_context *ctx, const camera &cam, int nx, int ny) { return rt_camera_set(ctx, &cam.desc, nx, ny); }

/* ---- octree (acceleration_structure.h:11-61): the reference's own memory layout ------------------------------------------- */
#define CHILDREN_COUNT 8
#define TREE_HEIGHT 3
#define NUMBER_NODES (1 + CHILDREN_COUNT + CHILDREN_COUNT * CHILDREN_COUNT + CHILDREN_COUNT * CHILDREN_COUNT * CHILDREN_COUNT)
#define NUMBER_LEAFS (CHILDREN_COUNT * CHILDREN_COUNT * CHILDREN_COUNT * CHILDREN_COUNT)
#ifndef SPHERES_PER_LEAF
#define SPHERES_PER_LEAF 30          /* acceleration_structure.h:15; -D overrides it, as the CLI does */
#endif
#ifdef USE_FP16
/* one real_t member of the USE_FP16 layout: the 2 bytes of an IEEE half, read as float */
struct rt_half_storage {
    uint16_t bits;
    operator float() const {
        const uint32_t sign = (uint32_t)(bits & 0x8000u) << 16, e = (bits >> 10) & 0x1fu, m = bits & 0x3ffu;
        uint32_t b;
        if (e == 0) {                                   /* zero or subnormal: m * 2^-24, exact in float */
            const float f = ldexpf((float)m, -24);
            memcpy(&b, &f, 4);
            b |= sign;
        } else if (e == 31) {
            b = sign | 0x7f800000u | (m << 13);         /* inf, NaN */
        } else {
            b = sign | ((e + 112u) << 23) | (m << 13);
        }
        float f;
        memcpy(&f, &b, 4);
        return f;
    }
};
struct AABB {                        /* acceleration_structure.h:26-29 with real_t = half: 12 bytes */
    rt_half_storage x_low, y_low, z_low;
    rt_half_storage x_high, y_high, z_high;
};
#else
struct AABB {
    real_t x_low, y_low, z_low;
    real_t x_high, y_high, z_high;
};
#endif
struct OctNode {
    int level;
    AABB aabb;
    int children[CHILDREN_COUNT];
};
struct OctLeaf {
    int sphere_indices[SPHERES_PER_LEAF];
    int index_count;
};
struct Octree {
    OctNode nodes[NUMBER_NODES];
    OctLeaf leaves[NUMBER_LEAFS + 1];
    int nodeCount = 0;
    int leafCount = 1;
};

/* acceleration_structure.h:195: the spheres become the bound context's world, the tree is built on the GPU (rt_octree_build)
 * and comes back in the reference layout, byte for byte what the serial host build produces.  nullptr on failure
 * (rt_last_error tells why).  The context keeps its own traversal structure for rendering and hitTree.  Under USE_FP16: the
 * tree of the FP16 build (half-rounded memberships, rt_octree_build_ex) in its layout. */
inline Octree *buildOctree(sphere *d_list, const int num_hitables) {
    rt_context *ctx = rt_dropin_context();
    if (!ctx || !d_list || num_hitables < 1) return nullptr;
    std::vector<rt_sphere_desc> flat;
    for (int i = 0; i < num_hitables; i++) d_list[i].flatten(flat);
    if (rt_scene_upload(ctx, flat.data(), num_hitables) != 0) return nullptr;
#ifdef USE_FP16
    if (rt_octree_build_ex(ctx, SPHERES_PER_LEAF, RT_PREC_FP16, nullptr) != 0) return nullptr;
    if (rt_octree_reference_bytes_ex(SPHERES_PER_LEAF, RT_PREC_FP16) != sizeof(Octree)) return nullptr;
#else
    if (rt_octree_build(ctx, SPHERES_PER_LEAF, nullptr) != 0) return nullptr;
    if (rt_octree_reference_bytes(SPHERES_PER_LEAF) != sizeof(Octree)) return nullptr;
#endif
    Octree *octree = new Octree();
    if (rt_octree_export_reference(ctx, octree, sizeof(Octree)) != 0) { delete octree; return nullptr; }
    return octree;
}

/* acceleration_structure.h:319: closest hit through the octree built by buildOctree (the `octree` argument names it; the
 * query runs on the context's own traversal structure, which returns the reference's answer).  `world` is the hitable_list
 * the spheres were uploaded from: it supplies mat_ptr for the record.  Under USE_FP16 the query is the FP16 build's and rec.t,
 * rec.p and rec.normal are its half values (sphere.h:30-33 as the library evaluates them, through rt_scatter_rays_ex with a
 * scratch state whose scattered ray is dropped). */
inline bool hitTree(Octree *octree, const ray &r, hit_record &rec, hitable **world) {
    rt_context *ctx = rt_dropin_context();
    if (!ctx || !octree) return false;
    const float o[3] = {r.A[0], r.A[1], r.A[2]}, d[3] = {r.B[0], r.B[1], r.B[2]};
    int idx = -1;
    float t = 0;
#ifdef USE_FP16
    if (rt_trace_rays_ex(ctx, 1, RT_PREC_FP16, 1, o, d, &idx, &t) != 0 || idx < 0) return false;
    uint32_t w[6] = {6615241u, 123456789u, 362436069u, 521288629u, 88675123u, 5783321u};    /* any non-zero XORWOW state */
    float p[3], nrm[3], od[3], att[3];
    int go = 0;
    if (rt_scatter_rays_ex(ctx, RT_PREC_FP16, 1, &idx, o, d, &t, w, p, nrm, od, att, &go) != 0 || go < 0) return false;
    rec.t = t;
    rec.sphere_index = idx;
    rec.p = vec3(p[0], p[1], p[2]);
    rec.normal = vec3(nrm[0], nrm[1], nrm[2]);
    rec.mat_ptr = nullptr;
    const hitable_list *wl = world ? dynamic_cast<const hitable_list *>(*world) : nullptr;
    const sphere *sp = (wl && idx < wl->list_size) ? dynamic_cast<const sphere *>(wl->list[idx]) : nullptr;
    if (sp) rec.mat_ptr = sp->mat_ptr;
    return true;
#else
    if (rt_trace_rays(ctx, 1, 1, o, d, &idx, &t) != 0 || idx < 0) return false;
    rec.t = t;
    rec.sphere_index = idx;
    rec.p = r.point_at_parameter(t);
    rec.mat_ptr = nullptr;
    const hitable_list *wl = world ? dynamic_cast<const hitable_list *>(*world) : nullptr;
    const sphere *sp = (wl && idx < wl->list_size) ? dynamic_cast<const sphere *>(wl->list[idx]) : nullptr;
    if (sp) { rec.mat_ptr = sp->mat_ptr; rec.normal = (rec.p - sp->center) / sp->radius; }
    return true;
#endif
}

#endif
