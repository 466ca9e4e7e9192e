// rt_trace.cuh — closest-hit queries: flat list (hitable_list.h:16-31) and octree (acceleration_structure.h:226-342).
//
// Result contract (SURVEY D10): the closest hit is the minimum over a CANDIDATE SET, with strict '<', so it does not
// depend on the order candidates are tested in, nor on testing candidates that cannot win.
//   flat list : candidate set = all spheres.
//   octree    : candidate set = ground sphere (index 0) + the stored lists of every level-3 cell whose reference
//               AABB passes the reference's infinite-LINE slab test (intersect_ray_aabb, :226-244, evaluated here
//               with the same float operations).  A parent box contains its children and float subtraction and
//               division are monotone, so a passing cell implies passing ancestors.
// The octree query never walks the tree.  Candidates come from one uniform grid over the small spheres, walked
// with a 3D-DDA in a single flat loop (every lane of a warp executes the same advance / test body, which is what
// keeps the warp converged), plus a short list of big spheres.  A candidate that would become the closest hit is
// accepted only if one of the cells that store it passes the reference's line test (VisView) — that reproduces the
// reference's quirks exactly: spheres dropped on bucket overflow, spheres outside the root box, hits the line test
// never reaches.  All pruning is conservative (margins below), so the minimum is unchanged.
#pragma once
#include <string.h>

#include "rt_shade.cuh"

namespace rt {

#if defined(__CUDA_ARCH__)
#define RT_LDG(p) __ldg(p)
#else
#define RT_LDG(p) (*(p))
#endif

// A float-evaluated root can sit this far (relative, along the ray) from where exact arithmetic would put it:
// near-tangent hits lose half the mantissa in sqrt(b*b - a*c).  Pruning keeps this much slack.
constexpr float kTSlackRel = 4e-3f;
constexpr float kTSlackAbs = 1e-3f;

struct Hit {
    float t;
    int idx;
};

// Work counters of the instrumented build (-DRT_COUNTERS -> librt_b200_counters.so); compiled out otherwise.
struct TraceCounters {
    uint32_t sphere_tests, node_tests, voxel_steps;
};
#ifdef RT_COUNTERS
#define RT_COUNT(field) (tc.field++)
#else
#define RT_COUNT(field) ((void)0)
#endif

// Ties: two DIFFERENT spheres with bit-identical t (~170 pixels of BASELINE config 3 at full size: 1e9 rays against 7-fold
// overlapping spheres).  The reference keeps whichever it tests FIRST (strict '<'): the ground sphere, then the level-3 cells
// in child order (= ascending 9-bit Morton id) whose boxes the ray's line crosses, each cell's leaf lists in ascending sphere
// index.  A tied sphere's place in that order is tie_key() = (first crossed cell that stores it, its index); the frame of the
// reference's CUDA build settles it (tests/golden/ref_cuda/manifest_full.json: with "smaller index wins" 21 pixels of that
// frame differ, with this rule none).  The closest-hit kernels only DETECT a tie (a candidate whose root equals the current
// minimum but whose index differs) and leave the decision to resolve_ties(): one more walk for ~1e-7 of the rays.
// tie_bound(t) is the next float above t, so that sphere_test's strict `root < t_max` lets an equal root through.
RT_HD float tie_bound(const float t) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(__float_as_uint(t) + 1u);
#else
    uint32_t u;
    memcpy(&u, &t, 4);
    u += 1u;
    float r;
    memcpy(&r, &u, 4);
    return r;
#endif
}

// ---- flat list: every sphere, SoA float4, warp-uniform address (broadcast) ------------------------------------
template <typename GeomPtr>
RT_HD Hit trace_list(const GeomPtr geom, const int *tag, const int n, const vec3f o, const vec3f d, TraceCounters &tc) {
    Hit h;
    h.t = kTMax; h.idx = -1;
    const float a = dot3(d, d);
    for (int i = 0; i < n; i++) {
        const float4 s = geom[i];
        float t;
        RT_COUNT(sphere_tests);
        // slots create_world never wrote carry radius 0 and tag NONE: skipped (SURVEY D3)
        if (sphere_test(s, o, d, a, h.t, t) && RT_LDG(tag + i) >= 0) { h.t = t; h.idx = i; }
    }
    return h;
}

// acceleration_structure.h:226-244 — same operations, same comparisons (NaN compares false as there)
RT_HD bool ref_line_test(const vec3f o, const vec3f d, const float xl, const float yl, const float zl, const float xh,
                         const float yh, const float zh) {
    float tmin = div_(sub_(xl, o.x), d.x), tmax = div_(sub_(xh, o.x), d.x);
    if (tmin > tmax) { const float t = tmin; tmin = tmax; tmax = t; }
    float tymin = div_(sub_(yl, o.y), d.y), tymax = div_(sub_(yh, o.y), d.y);
    if (tymin > tymax) { const float t = tymin; tymin = tymax; tymax = t; }
    if ((tmin > tymax) || (tymin > tmax)) return false;
    if (tymin > tmin) tmin = tymin;
    if (tymax < tmax) tmax = tymax;
    float tzmin = div_(sub_(zl, o.z), d.z), tzmax = div_(sub_(zh, o.z), d.z);
    if (tzmin > tzmax) { const float t = tzmin; tzmin = tzmax; tzmax = t; }
    if ((tmin > tzmax) || (tzmin > tmax)) return false;
    return true;
}

// 1/x for the TRAVERSAL only (grid clipping and DDA parameters; never an image value): the approximate reciprocal is good
// to 1 ulp, i.e. ~3e-6 in t at scene scale, against voxel lists padded by >= 2e-4 (rt_build.cuh sphere_pad) and the
// slack of ray_box; IEEE division costs ~10 instructions and a slow-path branch per component.
RT_HD float rcp_trav(const float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return 1.0f / x;
#endif
}

RT_HD float sqrt_trav(const float x) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return sqrtf(x);
#endif
}

// sphere.h:18-23 up to the discriminant (the same fused operations as sphere_test, so the compiler shares them), then a
// conservative pre-filter in front of the IEEE sqrt and divisions: both roots are estimated with approximate arithmetic;
// `true` means an estimate is within its error bound of the accepted interval (kTMin, t_max) and the exact evaluation
// must decide.  Error bound: reciprocal and square root good to 2^-22 plus three roundings keep |estimate - float root|
// below 3e-6 * (|b| + sqrt(disc)) / a; the filter allows 1e-5.  A NaN discriminant is not > 0: no candidate, as in
// sphere_test.  ia = rcp_trav(a).  Branch-free on purpose: the lanes of a warp test unrelated spheres.
RT_HD bool maybe_hit(const float4 s, const vec3f o, const vec3f d, const float a, const float ia, const float t_max) {
    const vec3f oc = mk(sub_(o.x, s.x), sub_(o.y, s.y), sub_(o.z, s.z));
    const float b = dot3(oc, d);
    const float c = fma_(-s.w, s.w, dot3(oc, oc));
    const float disc = fma_(b, b, -mul_(a, c));
    const float sa = sqrt_trav(fmaxf(disc, 0.0f));
    const float t1 = (-b - sa) * ia, t2 = (sa - b) * ia;
    const float eps = (fabsf(b) + sa) * ia * 1e-5f;
    const bool reject = (t1 - eps > t_max) | (t2 + eps < kTMin) | ((t1 + eps < kTMin) & (t2 - eps > t_max));
    return (disc > 0.0f) & !reject;
}

// The same pre-filter, and — when the estimates make a hit CERTAIN — an upper bound of the root sphere_test will accept:
// root1 surely above kTMin (accepted: root1 <= t1 + eps), or root1 surely below kTMin and root2 surely above it (accepted:
// root2 <= t2 + eps).  FLT_MAX otherwise (no hit, or the estimates straddle kTMin).  The closest hit of the ray is then at most
// `ub`, whatever the exact evaluation returns: the cooperative kernel prunes against it long before it evaluates exactly.
RT_HD bool maybe_hit_ub(const float4 s, const vec3f o, const vec3f d, const float a, const float ia, const float t_max, float &ub) {
    const vec3f oc = mk(sub_(o.x, s.x), sub_(o.y, s.y), sub_(o.z, s.z));
    const float b = dot3(oc, d);
    const float c = fma_(-s.w, s.w, dot3(oc, oc));
    const float disc = fma_(b, b, -mul_(a, c));
    const float sa = sqrt_trav(fmaxf(disc, 0.0f));
    const float t1 = (-b - sa) * ia, t2 = (sa - b) * ia;
    const float eps = (fabsf(b) + sa) * ia * 1e-5f;
    const float lo1 = t1 - eps, hi1 = t1 + eps, lo2 = t2 - eps, hi2 = t2 + eps;
    const bool reject = (lo1 > t_max) | (hi2 < kTMin) | ((hi1 < kTMin) & (lo2 > t_max));
    const bool pass = (disc > 0.0f) & !reject;
    float u = kTMax;
    if (lo1 > kTMin) u = hi1;
    else if ((hi1 < kTMin) & (lo2 > kTMin)) u = hi2;
    ub = pass ? u : kTMax;
    return pass;
}

struct RayPre {
    vec3f o, d, inv;    // inv = 1/d (IEEE; +-inf for zero components)
    float a;            // dot(d,d)
};

// Conservative ray/box interval: returns false when the ray cannot be inside [lo,hi] for any t in
// (kTMin, t_far].  fminf/fmaxf drop NaNs (0*inf), which only ever widens the interval.
RT_HD bool ray_box(const RayPre &r, const float *lo, const float *hi, const float t_far, float &t_enter, float &t_exit) {
    const float tx0 = (lo[0] - r.o.x) * r.inv.x, tx1 = (hi[0] - r.o.x) * r.inv.x;
    const float ty0 = (lo[1] - r.o.y) * r.inv.y, ty1 = (hi[1] - r.o.y) * r.inv.y;
    const float tz0 = (lo[2] - r.o.z) * r.inv.z, tz1 = (hi[2] - r.o.z) * r.inv.z;
    const float t0 = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    const float t1 = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), t_far));
    t_enter = t0;
    t_exit = t1;
    // slack: the box is padded at build time; this covers the rounding of the products above
    return t0 <= t1 * (1.0f + 1e-5f) + 1e-6f;
}

// 9-bit Morton id (3 bits per level, x bit highest — the child index of acceleration_structure.h:150-165) -> cell coords
RT_HD void cell_xyz(const int m, int &ix, int &iy, int &iz) {
    ix = ((m >> 8) & 1) << 2 | ((m >> 5) & 1) << 1 | ((m >> 2) & 1);
    iy = ((m >> 7) & 1) << 2 | ((m >> 4) & 1) << 1 | ((m >> 1) & 1);
    iz = ((m >> 6) & 1) << 2 | ((m >> 3) & 1) << 1 | (m & 1);
}

// The reference's visibility rule for sphere `idx`: some level-3 cell that STORES it is crossed by the ray's line.
// `last_ok` caches the last cell that passed for this ray (neighbouring candidates mostly share it).
#if defined(__CUDA_ARCH__)
__device__ __noinline__
#else
inline
#endif
bool sphere_visible(const VisView vis, const float *planes, const int idx, const vec3f o, const vec3f d, int &last_ok,
                    TraceCounters &tc) {
    const uint32_t b = RT_LDG(vis.ent_off + idx), e = RT_LDG(vis.ent_off + idx + 1);
    for (uint32_t k = b; k < e; k++) {
        const int c = (int)RT_LDG(vis.ent_cell + k);
        if (c == last_ok) return true;
        if (c & kEntDropped) continue;                       // the reference never stored it there (:135)
        int ix, iy, iz;
        cell_xyz(c, ix, iy, iz);
        RT_COUNT(node_tests);
        if (ref_line_test(o, d, planes[ix], planes[kPlanes + iy], planes[2 * kPlanes + iz], planes[ix + 1],
                          planes[kPlanes + iy + 1], planes[2 * kPlanes + iz + 1])) {
            last_ok = c;
            return true;
        }
    }
    return false;
}

// Place of sphere `idx` in the reference's test order among spheres that tie (see "Ties" above): the first level-3 cell in child
// order that stores it and that the ray's line crosses, then the index; 0 for the ground sphere (tested before the tree),
// 0xffffffff when no such cell exists (the reference never tests it: not a candidate).  Flat-list mode: list order = index.
RT_HD uint32_t tie_key(const TreeView &tv, const float *planes, const int idx, const vec3f o, const vec3f d, TraceCounters &tc) {
    if (idx <= 0) return 0u;
    if (!tv.check_visibility) return (uint32_t)idx;
    uint32_t best = 0xffffffffu;
    const uint32_t b = RT_LDG(tv.vis.ent_off + idx), e = RT_LDG(tv.vis.ent_off + idx + 1);
    for (uint32_t k = b; k < e; k++) {
        const int c = (int)RT_LDG(tv.vis.ent_cell + k);
        if (c & kEntDropped) continue;
        const uint32_t key = (uint32_t)c << 22 | (uint32_t)idx;
        if (key >= best) continue;
        int ix, iy, iz;
        cell_xyz(c, ix, iy, iz);
        RT_COUNT(node_tests);
        if (ref_line_test(o, d, planes[ix], planes[kPlanes + iy], planes[2 * kPlanes + iz], planes[ix + 1], planes[kPlanes + iy + 1],
                          planes[2 * kPlanes + iz + 1]))
            best = key;
    }
    return best;
}

// A sufficient condition for the rule above that needs no division and no list: the hit point P = o + t*d lies on the
// ray's line, so if P is strictly inside some level-3 cell that stores the sphere, the line crosses that cell and the
// reference's slab test passes — PROVIDED the margins absorb its float rounding.  With P inside [lo + m, hi - m] per
// axis, the exact slab parameters bracket t with slack m/|d_i|; the reference's two roundings per parameter move each
// by at most 1.2e-7 * |plane - o_i|, and computing P here by at most 2.4e-7 * (|o_i| + |P_i|): m = 1e-4 + 4e-6 * (|o_i|
// + |P_i|) covers both many times over (zero direction components give -inf / +inf slabs, which pass).  The cell
// stores the sphere iff `intersects` (acceleration_structure.h:82-93: centre inside the box expanded by r, evaluated in
// float) held at every level — parents contain children and float add/sub are monotone, so the level-3 box decides —
// and the entry was not dropped on overflow (tv.no_drops).  The centre test uses its own margin for the rounding of
// lo - r and hi + r.  False only means "ask sphere_visible".
RT_HD bool visible_fast(const TreeView &tv, const float *planes, const float4 s, const vec3f o, const vec3f d, const float t) {
    if (!tv.no_drops) return false;
    const float P[3] = {o.x + t * d.x, o.y + t * d.y, o.z + t * d.z};
    const float O[3] = {o.x, o.y, o.z}, C[3] = {s.x, s.y, s.z};
    bool ok = true;
#pragma unroll
    for (int a = 0; a < 3; a++) {
        const float *pl = planes + a * kPlanes;
        int i = (int)((P[a] - pl[0]) * tv.cell_inv[a]);
        i = i < 0 ? 0 : (i > 7 ? 7 : i);
        const float lo = pl[i], hi = pl[i + 1];
        const float m = 1e-4f + 4e-6f * (fabsf(O[a]) + fabsf(P[a]));
        const float mc = 1e-4f + 4e-6f * (fabsf(lo) + fabsf(hi) + s.w);
        ok = ok && (P[a] >= lo + m) && (P[a] <= hi - m) && (C[a] > lo - s.w + mc) && (C[a] < hi + s.w - mc);
    }
    return ok;
}

// One pass over the candidates.
//   kWalkMin     : the plain minimum over all candidates; *tie is set when two different spheres share that minimum;
//   kWalkChecked : the visibility rule on every candidate before it may become the closest hit, ties by tie_key (always exact);
//   kWalkTies    : among the candidates whose accepted root is exactly t_tie, the first in the reference's order (idx -1: none).
enum : int { kWalkMin = 0, kWalkChecked = 1, kWalkTies = 2 };

// the candidate (t, idx) against the closest hit so far, per mode; key_h: tie_key of h.idx in kWalkTies (0xffffffff: none yet)
template <int MODE>
RT_HD void walk_accept(const TreeView &tv, const float *planes, const vec3f o, const vec3f d, const float t, const int idx, Hit &h,
                       uint32_t &key_h, bool *tie, int &last_ok, TraceCounters &tc) {
    if (MODE == kWalkMin) {
        if (t < h.t) { h.t = t; h.idx = idx; if (tie) *tie = false; }
        else if (idx != h.idx && tie) *tie = true;                       // equal root, another sphere: resolve_ties decides
    } else if (MODE == kWalkChecked) {
        if (t < h.t) {
            if (sphere_visible(tv.vis, planes, idx, o, d, last_ok, tc)) { h.t = t; h.idx = idx; }
        } else if (idx != h.idx) {
            if (tie_key(tv, planes, idx, o, d, tc) < tie_key(tv, planes, h.idx, o, d, tc)) h.idx = idx;
        }
    } else {
        if (t == h.t && idx != h.idx) {
            const uint32_t key = tie_key(tv, planes, idx, o, d, tc);
            if (key < key_h) { key_h = key; h.idx = idx; }
        }
    }
}

template <int MODE>
RT_HD Hit trace_walk(const SceneView &sc, const TreeView &tv, const float *planes, const vec3f o, const vec3f d,
                    TraceCounters &tc, const float t_tie = 0.0f, bool *tie = nullptr) {
    Hit h;
    h.t = MODE == kWalkTies ? t_tie : kTMax; h.idx = -1;
    uint32_t key_h = 0xffffffffu;
    if (tie) *tie = false;
    RayPre r;
    r.o = o; r.d = d;
    r.a = dot3(d, d);
    const float ia = rcp_trav(r.a);
    {   // ground sphere first, unconditionally (:322-332)
        float t;
        RT_COUNT(sphere_tests);
        if (sphere_test(RT_LDG(sc.geom), o, d, r.a, kTMax, t)) {
            if (MODE != kWalkTies) { h.t = t; h.idx = 0; }
            else if (t == t_tie) { h.idx = 0; key_h = 0u; }
        }
    }
    int last_ok = -1;
    for (int k = 1; k < tv.nprolog; k++) {   // big spheres: tested directly (prolog[0] is the ground sphere)
        const int idx = (int)RT_LDG(tv.prolog + k);
        float t;
        RT_COUNT(sphere_tests);
        const float4 s = RT_LDG(sc.geom + idx);
        if (maybe_hit(s, o, d, r.a, ia, h.t) && sphere_test(s, o, d, r.a, tie_bound(h.t), t))
            walk_accept<MODE>(tv, planes, o, d, t, idx, h, key_h, tie, last_ok, tc);
    }
    const GridView &g = tv.grid;
    if (g.nx == 0) return h;
    r.inv = mk(rcp_trav(d.x), rcp_trav(d.y), rcp_trav(d.z));
    float te, tx;
    if (!ray_box(r, g.org, g.hi, h.t * (1.0f + kTSlackRel) + kTSlackAbs, te, tx)) return h;

    // ---- 3D-DDA over the grid, one flat loop: every iteration = (advance to the next voxel if the current list is
    //      exhausted) + (one sphere test if the list is not empty) ----
    int ix = (int)floorf((o.x + d.x * te - g.org[0]) * g.inv_vs[0]);
    int iy = (int)floorf((o.y + d.y * te - g.org[1]) * g.inv_vs[1]);
    int iz = (int)floorf((o.z + d.z * te - g.org[2]) * g.inv_vs[2]);
    ix = imin(imax(ix, 0), g.nx - 1);
    iy = imin(imax(iy, 0), g.ny - 1);
    iz = imin(imax(iz, 0), g.nz - 1);
    const int sx = d.x >= 0.0f ? 1 : -1, sy = d.y >= 0.0f ? 1 : -1, sz = d.z >= 0.0f ? 1 : -1;
    // ray parameter at which the ray leaves the current voxel along each axis; an axis the ray does not move along
    // never advances
    float tmx = fabsf(d.x) > 0.0f ? (g.org[0] + (float)(ix + (sx > 0)) * g.vs[0] - o.x) * r.inv.x : kTMax;
    float tmy = fabsf(d.y) > 0.0f ? (g.org[1] + (float)(iy + (sy > 0)) * g.vs[1] - o.y) * r.inv.y : kTMax;
    float tmz = fabsf(d.z) > 0.0f ? (g.org[2] + (float)(iz + (sz > 0)) * g.vs[2] - o.z) * r.inv.z : kTMax;
    const float dtx = fabsf(g.vs[0] * r.inv.x), dty = fabsf(g.vs[1] * r.inv.y), dtz = fabsf(g.vs[2] * r.inv.z);
    uint32_t k, e;
    {
        RT_COUNT(voxel_steps);
        const uint2 v = RT_LDG(g.vox + ((size_t)(iz * g.ny + iy) * g.nx + ix));
        k = v.x; e = v.x + v.y;
    }
    int budget = g.nx + g.ny + g.nz + 4;       // hard bound on voxel steps: the loop always terminates
    bool walking = true;
    while (walking) {
        if (k >= e) {
            // step into the neighbour the ray enters next; t_in is where it enters
            float t_in;
            if (tmx <= tmy && tmx <= tmz) { t_in = tmx; ix += sx; tmx += dtx; walking = (unsigned)ix < (unsigned)g.nx; }
            else if (tmy <= tmz)          { t_in = tmy; iy += sy; tmy += dty; walking = (unsigned)iy < (unsigned)g.ny; }
            else                          { t_in = tmz; iz += sz; tmz += dtz; walking = (unsigned)iz < (unsigned)g.nz; }
            // a later voxel can only hold hits at t >= t_in (minus the float slack); also stop at the grid exit
            if (t_in > h.t * (1.0f + kTSlackRel) + kTSlackAbs || t_in > tx * (1.0f + 1e-5f) + 1e-6f || --budget < 0) walking = false;
            if (walking) {
                RT_COUNT(voxel_steps);
                const uint2 v = RT_LDG(g.vox + ((size_t)(iz * g.ny + iy) * g.nx + ix));
                k = v.x; e = v.x + v.y;
            }
        }
        if (walking && k < e) {
            // candidate geometry in list order (one dependent load; the index is only needed for a hit) and the
            // conservative pre-filter in front of the exact test: ~8 of a ray's candidates have a positive discriminant,
            // fewer than 2 can be the closest hit.  Two candidates per trip: their loads and filters are independent
            // (the second filter sees the closest hit as it was before the first candidate — a larger bound, still
            // conservative); the exact tests run in list order against the up-to-date bound.
            const bool two = k + 1 < e;
#if defined(__CUDA_ARCH__)
            const float4 s0 = RT_LDG(g.ref_geom + k), s1 = RT_LDG(g.ref_geom + (two ? k + 1 : k));
#else
            const float4 s0 = sc.geom[g.refs[k]], s1 = sc.geom[g.refs[two ? k + 1 : k]];
#endif
            const bool m0 = maybe_hit(s0, o, d, r.a, ia, h.t), m1 = two & maybe_hit(s1, o, d, r.a, ia, h.t);
            float t;
            RT_COUNT(sphere_tests);
            if (m0 && sphere_test(s0, o, d, r.a, tie_bound(h.t), t))
                walk_accept<MODE>(tv, planes, o, d, t, (int)RT_LDG(g.refs + k), h, key_h, tie, last_ok, tc);
            if (two) RT_COUNT(sphere_tests);
            if (m1 && sphere_test(s1, o, d, r.a, tie_bound(h.t), t))
                walk_accept<MODE>(tv, planes, o, d, t, (int)RT_LDG(g.refs + k + 1), h, key_h, tie, last_ok, tc);
            k += two ? 2u : 1u;
        }
    }
    return h;
}

// What every closest-hit kernel does with its minimum over ALL candidates (h, and whether two different spheres tied for it):
// ties go through one more walk that ranks the tied spheres in the reference's test order; then the reference's visibility rule
// ("some cell that stores the sphere is crossed by the ray's line") on the winner — invisible candidates are rare (hits outside
// the root box, spheres dropped on bucket overflow), so it is evaluated once, where the warp has reconverged, and only a
// failure redoes the walk with the rule (and the tie order) applied to every candidate.
// (the two rare continuations — ranking tied spheres, redoing the walk with the rule on every candidate — are out of line so
// that they cost the kernels no registers)
#if defined(__CUDA_ARCH__)
__device__ __noinline__
#else
inline
#endif
Hit finish_hit_slow(const SceneView &sc, const TreeView &tv, const float *planes, const vec3f o, const vec3f d, Hit h, const bool tie,
                    TraceCounters &tc) {
    if (tie) {
        const Hit w = trace_walk<kWalkTies>(sc, tv, planes, o, d, tc, h.t);
        if (w.idx >= 0) {                     // (tie_key found a crossed cell that stores it: visible)
            h.idx = w.idx;
            return h;
        }
    }                                         // none of the tied spheres is visible, or the winner is not:
    return trace_walk<kWalkChecked>(sc, tv, planes, o, d, tc);
}

RT_HD Hit finish_hit(const SceneView &sc, const TreeView &tv, const float *planes, const vec3f o, const vec3f d, const Hit h, const bool tie,
                    TraceCounters &tc) {
    if (tie) return finish_hit_slow(sc, tv, planes, o, d, h, true, tc);
    if (h.idx > 0 && tv.check_visibility && !visible_fast(tv, planes, RT_LDG(sc.geom + h.idx), o, d, h.t)) {
        int last_ok = -1;                    // (the ground sphere, index 0, is tested unconditionally by the reference)
        if (!sphere_visible(tv.vis, planes, h.idx, o, d, last_ok, tc)) return finish_hit_slow(sc, tv, planes, o, d, h, false, tc);
    }
    return h;
}

// acceleration_structure.h:319-342 hitTree, re-organised (see the header comment): candidates from the grid walk, then finish_hit.
RT_HD Hit trace_tree(const SceneView &sc, const TreeView &tv, const float *planes, const vec3f o, const vec3f d,
                    TraceCounters &tc) {
    bool tie = false;
    const Hit h = trace_walk<kWalkMin>(sc, tv, planes, o, d, tc, 0.0f, &tie);
    return finish_hit(sc, tv, planes, o, d, h, tie, tc);
}

}  // namespace rt
