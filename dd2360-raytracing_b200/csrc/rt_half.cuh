// rt_half.cuh — the USE_FP16 build of the reference (precision_types.h:8), per-lane device code.
//
// With USE_FP16 the reference's real_t is a struct around __half (precision_types.h:16-163): every vec3 / ray / sphere /
// material operation rounds to half, EXCEPT where C++ overload resolution quietly falls back to float — unary minus,
// `sqrt(x)` (float sqrtf), `pow`, `1.0/t`, float-literal-on-the-left expressions — and where the CUDA half intrinsics are
// themselves approximate (__hdiv = rcp.approx * x with a fix-up for tiny quotients, hsqrt / hrsqrt = MUFU on float).
// This file states that arithmetic explicitly, operation by operation.  Where each expression lands (half or float,
// fused or not) was read off the SASS of the reference headers compiled with -DUSE_FP16 for sm_100 (small probe kernels
// around sphere::hit, reflect, refract, scatter, get_ray, color's sky branch, render's pixel arithmetic):
//   * half multiply-adds are contracted exactly like the float ones (DESIGN.md §4): a*b+c*d -> fma(a,b,c*d),
//     x-a*b -> fma(-a,b,x), dot -> fma(z,z',fma(x,x',y*y'));
//   * sphere::hit's two roots are FLOAT expressions of half inputs: (-b - hsqrt(disc)) / a and (-b + sqrtf(disc)) / a
//     with IEEE float division, rounded to half on assignment (sphere.h:25,36);
//   * length() = half(sqrtf(float(dot))) (vec3.h:34), v / length() uses __hdiv (vec3.h:146);
//   * the ground sphere (radius 1000) overflows: r*r = 1e6 > 65504 -> c = inf -> discriminant -inf/NaN -> never hit
//     (SURVEY D9): the FP16 image has no ground, by construction, here as there.
// The same intrinsics are used as in the reference build (__hdiv, hsqrt, hrsqrt, hsin, hcos), so their approximation
// errors are reproduced rather than modelled.  Vector operations are packed: (x, y) in one __half2, z separate —
// per-lane rounding of the packed instructions is identical to the scalar ones.
#pragma once
#include <cuda_fp16.h>

#include "rt_math.cuh"
#include "rt_types.h"

namespace rt {
namespace h16 {

typedef __half hf;

__device__ __forceinline__ hf f2h(float f) { return __float2half_rn(f); }
__device__ __forceinline__ float h2f(hf h) { return __half2float(h); }
__device__ __forceinline__ hf hfma_(hf a, hf b, hf c) { return __hfma(a, b, c); }
__device__ __forceinline__ hf hmul_(hf a, hf b) { return __hmul_rn(a, b); }
__device__ __forceinline__ hf hadd_(hf a, hf b) { return __hadd_rn(a, b); }
__device__ __forceinline__ hf hsub_(hf a, hf b) { return __hsub_rn(a, b); }
__device__ __forceinline__ hf hdiv_(hf a, hf b) { return __hdiv(a, b); }                 // real_t::operator/ (precision_types.h:56-63)
__device__ __forceinline__ hf hsqrtf_(hf a) { return f2h(__fsqrt_rn(h2f(a))); }          // sqrt(real_t) -> float sqrtf -> real_t
__device__ __forceinline__ hf hneg_(hf a) { return __hneg(a); }
// col /= real_t(ns): k = 1.0 / t in double, stored as real_t (vec3.h:137-144).  The one definition of the divisor of the final
// average: k_render_h and k_finalize_h both use it, so a frame finalised from shards or progressive sums is the one-shot frame.
__device__ __forceinline__ hf inv_ns_h(int ns) { return f2h((float)(1.0 / (double)h2f(f2h((float)ns)))); }

struct vec3h {
    __half2 xy;
    hf z;
};
__device__ __forceinline__ vec3h mkh(hf x, hf y, hf z) { vec3h v; v.xy = __halves2half2(x, y); v.z = z; return v; }
__device__ __forceinline__ vec3h mkh_f(float x, float y, float z) { return mkh(f2h(x), f2h(y), f2h(z)); }
__device__ __forceinline__ hf vx(const vec3h v) { return __low2half(v.xy); }
__device__ __forceinline__ hf vy(const vec3h v) { return __high2half(v.xy); }
__device__ __forceinline__ vec3h vsub(const vec3h a, const vec3h b) { vec3h r; r.xy = __hsub2_rn(a.xy, b.xy); r.z = hsub_(a.z, b.z); return r; }
__device__ __forceinline__ vec3h vadd(const vec3h a, const vec3h b) { vec3h r; r.xy = __hadd2_rn(a.xy, b.xy); r.z = hadd_(a.z, b.z); return r; }
__device__ __forceinline__ vec3h vmul(const vec3h a, const vec3h b) { vec3h r; r.xy = __hmul2_rn(a.xy, b.xy); r.z = hmul_(a.z, b.z); return r; }
__device__ __forceinline__ vec3h vscale(const hf t, const vec3h a) { vec3h r; r.xy = __hmul2_rn(__half2half2(t), a.xy); r.z = hmul_(t, a.z); return r; }
// a * t + c per component
__device__ __forceinline__ vec3h vfma(const vec3h a, const hf t, const vec3h c) { vec3h r; r.xy = __hfma2(a.xy, __half2half2(t), c.xy); r.z = hfma_(a.z, t, c.z); return r; }
__device__ __forceinline__ vec3h vneg(const vec3h a) { vec3h r; r.xy = __hneg2(a.xy); r.z = hneg_(a.z); return r; }

// vec3.h:91-93 dot(): fma(z,z', fma(x,x', y*y'))
__device__ __forceinline__ hf dot3h(const vec3h a, const vec3h b) { return hfma_(a.z, b.z, hfma_(vx(a), vx(b), hmul_(vy(a), vy(b)))); }
// vec3.h:34 length(): the squares in half, the root in float
__device__ __forceinline__ hf lengthh(const vec3h v) { return hsqrtf_(dot3h(v, v)); }
// vec3.h:146-148 unit_vector(): v / v.length(), three __hdiv
__device__ __forceinline__ vec3h unit_vectorh(const vec3h v) {
    const hf len = lengthh(v);
    return mkh(hdiv_(vx(v), len), hdiv_(vy(v), len), hdiv_(v.z, len));
}

__device__ __forceinline__ hf uniform_h(xorwow &s) { return f2h(xorwow_uniform(s)); }   // curand_uniform() is float; real_t(float) rounds

struct SphereH {            // one sphere in half: what the FP16 create_world stores (the FP32 scene rounded once)
    vec3h c;
    hf r;
};
__device__ __forceinline__ SphereH load_sphere_h(const uint2 *geom_h, int i) {
    const uint2 u = __ldg(geom_h + i);
    SphereH s;
    s.c.xy = *reinterpret_cast<const __half2 *>(&u.x);
    const __half2 zr = *reinterpret_cast<const __half2 *>(&u.y);
    s.c.z = __low2half(zr);
    s.r = __high2half(zr);
    return s;
}

// sphere.h:17-46 under USE_FP16.  t_min = real_t(0.001f); returns true and the accepted root when t_min < t < t_max.
__device__ __forceinline__ bool sphere_test_h(const SphereH s, const vec3h o, const vec3h d, const hf a, const hf t_max, hf &t_out) {
    const vec3h oc = vsub(o, s.c);                                        // sphere.h:18
    const hf b = dot3h(oc, d);                                            // :20
    const hf c = hfma_(hneg_(s.r), s.r, dot3h(oc, oc));                   // :21
    const hf disc = hfma_(b, b, hneg_(hmul_(a, c)));                      // :22
    if (__hgt(disc, f2h(0.0f))) {
        const float fb = h2f(b), fa = h2f(a);
        const hf t_min = f2h(0.001f);
        hf temp = f2h(__fdiv_rn(__fsub_rn(-fb, h2f(hsqrt(disc))), fa));   // :25  (-b - real_t::sqrt(disc)) / a  in float
        if (__hlt(temp, t_max) && __hgt(temp, t_min)) { t_out = temp; return true; }
        temp = f2h(__fdiv_rn(__fadd_rn(-fb, __fsqrt_rn(h2f(disc))), fa));  // :36  (-b + sqrt(disc)) / a        in float
        if (__hlt(temp, t_max) && __hgt(temp, t_min)) { t_out = temp; return true; }
    }
    return false;
}

// sphere.h:30-33: p = A + t*B (fused), normal = (p - center) / radius (__hdiv)
__device__ __forceinline__ void hit_point_h(const SphereH s, const vec3h o, const vec3h d, const hf t, vec3h &p, vec3h &n) {
    p = vfma(d, t, o);
    const vec3h pc = vsub(p, s.c);
    n = mkh(hdiv_(vx(pc), s.r), hdiv_(vy(pc), s.r), hdiv_(pc.z, s.r));
}

// material.h:33-41: p = real_t(2)*RANDVEC3 - vec3(1,1,1) until squared_length() < 1
__device__ __forceinline__ vec3h random_in_unit_sphere_h(xorwow &rng) {
    vec3h p;
    const hf two = f2h(2.0f), m1 = f2h(-1.0f);
    do {
        const hf u0 = uniform_h(rng), u1 = uniform_h(rng), u2 = uniform_h(rng);
        p = mkh(hfma_(u0, two, m1), hfma_(u1, two, m1), hfma_(u2, two, m1));
    } while (__hge(dot3h(p, p), f2h(1.0f)));
    return p;
}

// material.h:43-45 reflect: v - real_t(2)*dot(v,n)*n
__device__ __forceinline__ vec3h reflect_h(const vec3h v, const vec3h n) {
    const hf d2 = hmul_(dot3h(v, n), f2h(2.0f));
    return vfma(n, hneg_(d2), v);
}

// material.h:17-31 refract
__device__ __forceinline__ bool refract_h(const vec3h v, const vec3h n, const hf ni_over_nt, vec3h &refracted) {
    const vec3h uv = unit_vectorh(v);
    const hf dt = dot3h(uv, n);
    const hf one = f2h(1.0f);
    const hf disc = hfma_(hneg_(hmul_(ni_over_nt, ni_over_nt)), hfma_(hneg_(dt), dt, one), one);
    if (__hgt(disc, f2h(0.0f))) {
        const hf sq = hsqrt(disc);                                           // real_t::sqrt -> hsqrt (:24)
        const vec3h inner = vfma(n, hneg_(dt), uv);                          // uv - n*dt
        // ni*(uv - n*dt) - n*sq: here ptxas fuses the LEFT product, fma(inner, ni, -(sq*n)) (FP32 fuses the right one)
        const vec3h nsq = vscale(sq, n);
        refracted = vfma(inner, ni_over_nt, vneg(nsq));
        return true;
    }
    return false;
}

// material.h:11-15 schlick: (1 -/+ ref_idx) and pow() are float, the rest half
__device__ __forceinline__ hf schlick_h(const hf cosine, const hf ref_idx) {
    hf r0 = hdiv_(f2h(1.0f - h2f(ref_idx)), f2h(1.0f + h2f(ref_idx)));
    r0 = hmul_(r0, r0);
    return hfma_(f2h(1.0f - h2f(r0)), f2h(powf(1.0f - h2f(cosine), 5.0f)), r0);
}

struct MatH {
    vec3h albedo;
    hf param;       // metal: fuzz (clamped to <= 1 by metal::metal, material.h:66); dielectric: ref_idx
};
__device__ __forceinline__ MatH load_mat_h(const uint2 *matl_h, int i) {
    const uint2 u = __ldg(matl_h + i);
    MatH m;
    m.albedo.xy = *reinterpret_cast<const __half2 *>(&u.x);
    const __half2 zp = *reinterpret_cast<const __half2 *>(&u.y);
    m.albedo.z = __low2half(zp);
    m.param = __high2half(zp);
    return m;
}

// material.h:55-60 / :68-73 / :81-113 under USE_FP16; returns false when the ray is absorbed (metal only)
__device__ __forceinline__ bool scatter_h(const int tag, const MatH m, const vec3h d_in, const vec3h p, const vec3h n, vec3h &atten,
                                          vec3h &d_out, xorwow &rng) {
    if (tag == 0) {
        const vec3h r = random_in_unit_sphere_h(rng);
        const vec3h target = vadd(vadd(p, n), r);
        d_out = vsub(target, p);
        atten = m.albedo;
        return true;
    }
    if (tag == 1) {
        const vec3h refl = reflect_h(unit_vectorh(d_in), n);
        const vec3h r = random_in_unit_sphere_h(rng);
        d_out = vfma(r, m.param, refl);                                      // reflected + fuzz*r
        atten = m.albedo;
        return __hgt(dot3h(d_out, n), f2h(0.0f));
    }
    const hf ref_idx = m.param, one = f2h(1.0f);
    const vec3h reflected = reflect_h(d_in, n);
    vec3h outward, refracted = mkh_f(0.f, 0.f, 0.f);
    hf ni_over_nt, cosine, reflect_prob;
    atten = mkh(one, one, one);
    const hf ddn = dot3h(d_in, n);
    if (__hgt(ddn, f2h(0.0f))) {
        outward = vneg(n);
        ni_over_nt = ref_idx;
        cosine = hdiv_(ddn, lengthh(d_in));                                                       // real_t / real_t (:92)
        cosine = hsqrtf_(hfma_(hneg_(hmul_(ref_idx, ref_idx)), hfma_(hneg_(cosine), cosine, one), one));   // :93 sqrt() is float
    } else {
        outward = n;
        ni_over_nt = hdiv_(one, ref_idx);
        cosine = f2h(__fdiv_rn(-h2f(ddn), h2f(lengthh(d_in))));                                    // -dot is float, float / real_t is float (:98)
    }
    if (refract_h(d_in, outward, ni_over_nt, refracted)) reflect_prob = schlick_h(cosine, ref_idx);
    else reflect_prob = one;
    d_out = (xorwow_uniform(rng) < h2f(reflect_prob)) ? reflected : refracted;                    // float < real_t compares as float
    return true;
}

struct CameraH {
    vec3h origin, lower_left_corner, horizontal, vertical, u, v, w;
    hf lens_radius;
};
// the 22 halves k_camera_setup_h writes, in CameraData order (origin, llc, horizontal, vertical, u, v, w, lens_radius)
__device__ __forceinline__ CameraH load_camera_h(const __half *cam_h) {
    CameraH cam;
    vec3h *v[7] = {&cam.origin, &cam.lower_left_corner, &cam.horizontal, &cam.vertical, &cam.u, &cam.v, &cam.w};
    for (int k = 0; k < 7; k++) *v[k] = mkh(cam_h[3 * k], cam_h[3 * k + 1], cam_h[3 * k + 2]);
    cam.lens_radius = cam_h[21];
    return cam;
}

// camera.h:12-18 + :45-49 under USE_FP16
__device__ __forceinline__ void camera_ray_h(const CameraH &c, const hf s, const hf t, xorwow &rng, vec3h &o, vec3h &d) {
    hf px, py;
    const hf two = f2h(2.0f), m1 = f2h(-1.0f);
    do {
        const hf u0 = uniform_h(rng), u1 = uniform_h(rng);
        px = hfma_(u0, two, m1);
        py = hfma_(u1, two, m1);
    } while (__hge(hfma_(px, px, hmul_(py, py)), f2h(1.0f)));       // dot(p,p) with p.z = 0: the z term adds an exact zero
    const hf rdx = hmul_(c.lens_radius, px), rdy = hmul_(c.lens_radius, py);
    const vec3h off = vfma(c.u, rdx, vscale(rdy, c.v));            // u*rd.x + v*rd.y
    o = vadd(c.origin, off);
    d = vsub(vsub(vfma(c.vertical, t, vfma(c.horizontal, s, c.lower_left_corner)), c.origin), off);
}

// main.cu:68-71 under USE_FP16: (1.0f - t) is a float subtraction rounded to half
__device__ __forceinline__ vec3h sky_h(const vec3h d) {
    const vec3h ud = unit_vectorh(d);
    const hf t = hmul_(hadd_(vy(ud), f2h(1.0f)), f2h(0.5f));
    const hf omt = f2h(1.0f - h2f(t));
    return mkh(hfma_(t, f2h(0.5f), omt), hfma_(t, f2h(0.7f), omt), hadd_(omt, t));
}

// acceleration_structure.h:226-244 under USE_FP16: AABB members, ray origin and direction are real_t, so every slab
// parameter is (half - half) / half with __hdiv, widened to float only for the comparisons
__device__ __forceinline__ bool ref_line_test_h(const vec3h o, const vec3h d, const hf xl, const hf yl, const hf zl, const hf xh,
                                                const hf yh, const hf zh) {
    float tmin = h2f(hdiv_(hsub_(xl, vx(o)), vx(d))), tmax = h2f(hdiv_(hsub_(xh, vx(o)), vx(d)));
    if (tmin > tmax) { const float t = tmin; tmin = tmax; tmax = t; }
    float tymin = h2f(hdiv_(hsub_(yl, vy(o)), vy(d))), tymax = h2f(hdiv_(hsub_(yh, vy(o)), vy(d)));
    if (tymin > tymax) { const float t = tymin; tymin = tymax; tymax = t; }
    if ((tmin > tymax) || (tymin > tmax)) return false;
    if (tymin > tmin) tmin = tymin;
    if (tymax < tmax) tmax = tymax;
    float tzmin = h2f(hdiv_(hsub_(zl, o.z), d.z)), tzmax = h2f(hdiv_(hsub_(zh, o.z), d.z));
    if (tzmin > tzmax) { const float t = tzmin; tzmin = tzmax; tzmax = t; }
    if ((tmin > tzmax) || (tzmin > tmax)) return false;
    return true;
}

struct HitH {
    hf t;
    int idx;
};

// ---- candidate lists as PAIRS: two spheres per packed instruction ------------------------------------------------------------
// A list (all spheres for the flat mode, the stored list of one level-3 cell for the octree) is laid out as pairs of
// consecutive candidates, transposed: {cx0,cx1} {cy0,cy1} {cz0,cz1} {r0,r1} = one 16-byte load, so that the discriminant
// of sphere.h:18-22 is evaluated for two spheres by each __half2 instruction (per-lane rounding of the packed
// instructions is that of the scalar ones, so the two discriminants are bit-identical to sphere_test_h's).  Only when
// one of them is positive is the scalar root evaluation run — in list order, because exact ties between different
// spheres are common with 11 significant bits and the reference keeps the first.  Slots create_world never wrote
// (tag NONE) are left out when the pairs are built; an odd tail is padded with a NaN sphere (discriminant NaN: never > 0).
struct PairView {
    const uint4 *geom;        // transposed pair geometry
    const int2 *idx;          // the two sphere indices (-1: padding)
    const uint32_t *start;    // pairs of list m: [start[m], start[m+1])
};

// Semantics the cooperative scan below reproduces:
//   flat list (hitable_list.h:16-31): every sphere in ascending index order, strict '<' against closest_so_far;
//   octree (acceleration_structure.h:276-342): ground sphere first, then the tree in the reference's own order — children
//   by octant index at every level (= ascending Morton code), the stored list of each level-3 cell in insertion
//   (= ascending sphere index) order — with the half-precision line test at EVERY level (approximate __hdiv is not
//   monotone, so a child's pass does not imply its parent's); entries beyond 8*SPL per cell were dropped (:135).
//   No sub-grid: in half arithmetic a sphere can "hit" far from where it is, so every sphere of a passing cell is a real
//   candidate, exactly as in the reference.

// ---- warp-cooperative closest hit ---------------------------------------------------------------------------------------------
// The USE_FP16 closest hit is an exhaustive scan (every sphere of every passing cell: ~2 000 candidates per ray at 100 k
// spheres), so instead of 32 lanes each crawling through their own lists, the WARP takes the rays of its lanes one at a
// time: the ray is broadcast, the lanes test the existing octree nodes compacted (root + level 1 in one warp step, level 2
// in one, level 3 only for the children of the level-2 nodes that passed, four parents per step), then stride through the
// pair list of each passing cell together — coalesced 16-byte loads, no divergence.  The scan only FILTERS (four pair loads
// in flight per lane, packed discriminants) and pushes the positives, as scan-order keys, into a ring in shared memory;
// whenever 32 keys are queued, the 32 lanes evaluate one candidate each, converged.  (About 6 % of the candidates of a
// passing cell have a positive discriminant: evaluated inside the scan loop, the ~150 instructions of two scalar sphere
// tests with IEEE sqrt / div ran under a branch that a few lanes take in nearly every iteration, and dominated the ~20 of
// the filter.)  Equivalence with the reference's sequential scan: a candidate's accepted root t_i does not depend on
// closest_so_far (if the near root is valid but not closer, the far root is not closer either), so the sequential result
// is the lexicographic minimum of (t_i, position in scan order) — ties keep the first, as strict '<' does.  That minimum
// does not depend on the order candidates are evaluated in; it is taken with two warp-wide REDUX mins.
struct NodeTab {
    const uint2 *ent;         // [8 | 64 | 512] compact per level: x = ix | iy << 8 | iz << 16, y = parent position | morton << 16
    const uint32_t *count;    // n1, n2, n3
};

struct BestH {                // lane-local lexicographic minimum of (t bits, scan position)
    uint32_t t, order;
};
__device__ __forceinline__ void best_update(BestH &b, const hf t, const uint32_t order) {
    const uint32_t tb = __half_as_ushort(t);          // accepted roots are > 0.001: positive halves order like their bits
    if (tb < b.t || (tb == b.t && order < b.order)) { b.t = tb; b.order = order; }
}

constexpr uint32_t kPairPad = 128;      // every pair list is padded with NaN pairs to a multiple of this (k_pairs_fill)
struct CoopSmem {
    uint32_t ring[512];       // scan-order keys of candidates with a positive discriminant (0: the ground sphere)
    uint32_t cells[16][32];   // scratch: the compacted list of the level-2 nodes a ray passes (coop_trace_h)
    uint32_t tail;            // ring write position (shared atomic: the order of the keys in the ring does not matter)
    uint32_t pairs_lo, pairs_hi;   // RT_COUNTERS builds: sphere pairs scanned by this warp (work counter of the roofline)
    uint32_t pad_;
};

__device__ __forceinline__ void coop_eval_h(const PairView pv, const uint2 *geom_h, const uint32_t key, const vec3h o, const vec3h d, const hf a,
                                            BestH &best) {
    SphereH s;
    if (key == 0u) {
        s = load_sphere_h(geom_h, 0);
    } else {
        const uint32_t k = (key - 1u) >> 1, sel = ((key - 1u) & 1u) * 16u;
        const uint4 g = __ldg(pv.geom + k);
        s.c = mkh(__ushort_as_half((unsigned short)(g.x >> sel)), __ushort_as_half((unsigned short)(g.y >> sel)),
                  __ushort_as_half((unsigned short)(g.z >> sel)));
        s.r = __ushort_as_half((unsigned short)(g.w >> sel));
    }
    hf t;
    if (sphere_test_h(s, o, d, a, f2h(3.402823466e+38f), t)) best_update(best, t, key);
}

// evaluate the queued candidates 32 at a time, one per lane (everything that is left when `flush`); call converged
__device__ __forceinline__ void coop_drain_h(CoopSmem &sm, const PairView pv, const uint2 *geom_h, uint32_t &head, const bool flush,
                                             const unsigned lane, const vec3h o, const vec3h d, const hf a, BestH &best) {
    __syncwarp();
    const uint32_t tail = *reinterpret_cast<volatile uint32_t *>(&sm.tail);
    while (tail - head >= 32u || (flush && tail != head)) {
        const uint32_t left = tail - head;
        if (lane < left) coop_eval_h(pv, geom_h, sm.ring[(head + lane) & 511u], o, d, a, best);
        head += left < 32u ? left : 32u;
    }
    __syncwarp();
}

// all 32 lanes filter pairs [pb, pe) of one list (pe - pb a multiple of kPairPad) for the broadcast ray (o, d)
__device__ __forceinline__ void coop_filter_h(CoopSmem &sm, const PairView pv, const uint2 *geom_h, const uint32_t pb, const uint32_t pe,
                                              const unsigned lane, const vec3h o, const vec3h d, const hf a, uint32_t &head, BestH &best) {
    const unsigned full = 0xffffffffu;
    const __half2 ox = __half2half2(vx(o)), oy = __half2half2(vy(o)), oz = __half2half2(o.z);
    const __half2 dx = __half2half2(vx(d)), dy = __half2half2(vy(d)), dz = __half2half2(d.z);
    const __half2 a2 = __half2half2(a), zero2 = __float2half2_rn(0.0f);
    uint4 g[4];
#ifdef RT_COUNTERS
    if (lane == 0) {
        const uint32_t before = sm.pairs_lo;
        sm.pairs_lo = before + (pe - pb);
        if (sm.pairs_lo < before) sm.pairs_hi++;
    }
#endif
    if (pb < pe) {
#pragma unroll
        for (int i = 0; i < 4; i++) g[i] = __ldg(pv.geom + pb + lane + 32 * i);
    }
    for (uint32_t base = pb + lane; base < pe; base += kPairPad) {
        uint32_t mine = 0u;       // bit i: low sphere of pair i has a positive discriminant; bit 16 + i: its high sphere
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const __half2 cx = *reinterpret_cast<const __half2 *>(&g[i].x), cy = *reinterpret_cast<const __half2 *>(&g[i].y);
            const __half2 cz = *reinterpret_cast<const __half2 *>(&g[i].z), r = *reinterpret_cast<const __half2 *>(&g[i].w);
            const __half2 ocx = __hsub2_rn(ox, cx), ocy = __hsub2_rn(oy, cy), ocz = __hsub2_rn(oz, cz);            // sphere.h:18
            const __half2 b = __hfma2(ocz, dz, __hfma2(ocx, dx, __hmul2_rn(ocy, dy)));                               // :20
            const __half2 c = __hfma2(__hneg2(r), r, __hfma2(ocz, ocz, __hfma2(ocx, ocx, __hmul2_rn(ocy, ocy))));   // :21
            const __half2 disc = __hfma2(b, b, __hneg2(__hmul2_rn(a2, c)));                                          // :22
            mine |= __hgt2_mask(disc, zero2) & (0x00010001u << i);    // 0xffff per half where positive (NaN: 0)
        }
        if (base + kPairPad < pe) {      // the next step's loads fly while this step's positives are queued and evaluated
#pragma unroll
            for (int i = 0; i < 4; i++) g[i] = __ldg(pv.geom + base + kPairPad + 32 * i);
        }
        if (__any_sync(full, mine != 0u)) {
            while (mine) {                                           // ~0.5 positives per lane and step
                const uint32_t bit = (uint32_t)__ffs((int)mine) - 1u;
                mine &= mine - 1u;
                sm.ring[atomicAdd(&sm.tail, 1u) & 511u] = 2u * (base + 32u * (bit & 15u)) + 1u + (bit >> 4);
            }
            coop_drain_h(sm, pv, geom_h, head, false, lane, o, d, a, best);
        }
    }
}

// Closest hit of every lane's ray, one ray at a time by the whole warp.  The line tests of ray r are shared by the warp too
// (slab planes as halves in shared memory): a per-lane walk of the node tables measured 4 % (C4) to 20 % (488 spheres) slower.
template <bool OCTREE>
__device__ __forceinline__ HitH coop_trace_h(CoopSmem &sm, const hf *planes_h, const PairView pv, const NodeTab nt, const uint2 *geom_h,
                                             const bool have_ray, const vec3h o, const vec3h d) {
    const unsigned full = 0xffffffffu;
    const unsigned lane = threadIdx.x & 31u;
    HitH mine;
    mine.t = f2h(3.402823466e+38f);
    mine.idx = -1;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t n1 = 0, n2 = 0;
    if (OCTREE) { n1 = __ldg(nt.count); n2 = __ldg(nt.count + 1); }
    auto pass = [&](const uint32_t ex, const int level, const vec3h ro, const vec3h rd) {
        const int ix = ex & 255, iy = (ex >> 8) & 255, iz = (ex >> 16) & 255, sh = 3 - level;
        return ref_line_test_h(ro, rd, planes_h[ix << sh], planes_h[kPlanes + (iy << sh)], planes_h[2 * kPlanes + (iz << sh)],
                               planes_h[(ix + 1) << sh], planes_h[kPlanes + ((iy + 1) << sh)], planes_h[2 * kPlanes + ((iz + 1) << sh)]);
    };
    unsigned todo = __ballot_sync(full, have_ray);
    while (todo) {
        const int r = __ffs(todo) - 1;
        todo &= todo - 1u;
        vec3h ro, rd;
        {
            const uint32_t oxy = __shfl_sync(full, *reinterpret_cast<const uint32_t *>(&o.xy), r);
            const uint32_t dxy = __shfl_sync(full, *reinterpret_cast<const uint32_t *>(&d.xy), r);
            const __half2 zz = __halves2half2(o.z, d.z);
            const uint32_t ozdz = __shfl_sync(full, *reinterpret_cast<const uint32_t *>(&zz), r);
            ro.xy = *reinterpret_cast<const __half2 *>(&oxy);
            rd.xy = *reinterpret_cast<const __half2 *>(&dxy);
            const __half2 z2 = *reinterpret_cast<const __half2 *>(&ozdz);
            ro.z = __low2half(z2);
            rd.z = __high2half(z2);
        }
        const hf a = dot3h(rd, rd);
        BestH best;
        best.t = 0xffffffffu;
        best.order = 0xffffffffu;
        uint32_t head = *reinterpret_cast<volatile uint32_t *>(&sm.tail);       // the ring is empty between rays
        if (!OCTREE) {
            coop_filter_h(sm, pv, geom_h, __ldg(pv.start), __ldg(pv.start + 1), lane, ro, rd, a, head, best);   // hitable_list.h:16-31
        } else {
            if (lane == 0) { sm.ring[head & 511u] = 0u; sm.tail = head + 1u; }     // the ground sphere, tested unconditionally (:322-332)
            __syncwarp();                                                           // the other lanes' ring pushes (shared atomics) come after this store
            uint32_t *plist = &sm.cells[0][0];                                      // level-2 nodes that passed, compacted
            uint2 e = make_uint2(0u, 0u);
            if (lane >= 1u && lane <= n1) e = __ldg(nt.ent + lane - 1u);
            const unsigned m01 = __ballot_sync(full, lane <= n1 && pass(e.x, lane ? 1 : 0, ro, rd));
            const unsigned m1 = (n1 > 0 && (m01 & 1u)) ? m01 >> 1 : 0u;
            uint32_t np = 0;
            if (m1) {
                for (uint32_t b2 = 0; b2 < n2; b2 += 32u) {
                    const uint32_t j = b2 + lane;
                    const uint2 e2 = j < n2 ? __ldg(nt.ent + 8 + j) : make_uint2(0u, 0u);
                    const bool ok = j < n2 && ((m1 >> (e2.y & 0xffffu)) & 1u) && pass(e2.x, 2, ro, rd);
                    const unsigned m2 = __ballot_sync(full, ok);
                    if (ok) plist[np + __popc(m2 & lt)] = j;
                    np += __popc(m2);
                }
            }
            __syncwarp();
            for (uint32_t b3 = 0; b3 < np; b3 += 4u) {
                const uint32_t slot = b3 + (lane >> 3);
                uint2 e3 = make_uint2(0u, 0u);
                bool ok = false;
                if (slot < np) {
                    const uint32_t kid = __ldg(nt.count + 4 + plist[slot]);       // first child | count << 16
                    if ((lane & 7u) < (kid >> 16)) {
                        e3 = __ldg(nt.ent + 72 + (kid & 0xffffu) + (lane & 7u));
                        ok = pass(e3.x, 3, ro, rd);
                    }
                }
                unsigned m3 = __ballot_sync(full, ok);
                while (m3) {
                    const int c = __ffs(m3) - 1;
                    m3 &= m3 - 1u;
                    const uint32_t cell = __shfl_sync(full, e3.y >> 16, c);
                    coop_filter_h(sm, pv, geom_h, __ldg(pv.start + cell), __ldg(pv.start + cell + 1), lane, ro, rd, a, head, best);
                }
            }
            __syncwarp();
        }
        coop_drain_h(sm, pv, geom_h, head, true, lane, ro, rd, a, best);
        const uint32_t tmin = __reduce_min_sync(full, best.t);
        if (tmin != 0xffffffffu) {
            const uint32_t omin = __reduce_min_sync(full, best.t == tmin ? best.order : 0xffffffffu);
            if ((int)lane == r) {
                mine.t = __ushort_as_half((unsigned short)tmin);
                if (omin == 0u) {
                    mine.idx = 0;
                } else {
                    const int2 id = __ldg(pv.idx + ((omin - 1u) >> 1));
                    mine.idx = ((omin - 1u) & 1u) ? id.y : id.x;
                }
            }
        }
    }
    return mine;
}

}  // namespace h16
}  // namespace rt
