// hostsim.cpp — TEST-ONLY host emulation of the product's per-lane device code (never linked into librt_b200.so).
//
// The render kernel's arithmetic lives in __host__ __device__ headers (rt_shade.cuh, rt_trace.cuh, rt_build.cuh)
// whose float primitives map to explicitly rounded operations on both sides (rt_math.cuh).  Compiling them for
// the host lets the CPU-only test tier run the PRODUCT's closest-hit and shading code against the oracle without
// a GPU: it catches traversal / margin / arithmetic-pattern bugs before any GPU minute is spent.  What it cannot
// cover — the build kernels, the persistent scheduling, libdevice powf/tanf — is covered by the -m gpu tests.
//
// The traversal structure is rebuilt here on the host from a reference-layout Octree blob (so the candidate lists
// are exactly the reference's) using the same per-item functions the build kernels call (sphere_pad, choose_grid,
// voxel_range, shell_hits_box).  This is not a fallback path: the library has none.
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../dd2360-raytracing_b200/csrc/rt_build.cuh"
#include "../../dd2360-raytracing_b200/csrc/rt_trace.cuh"

using namespace rt;

static inline float4 make_float4(float x, float y, float z, float w) { float4 v; v.x = x; v.y = y; v.z = z; v.w = w; return v; }

struct hs_sphere { float cx, cy, cz, radius; int32_t mat; float ax, ay, az, param; };
struct hs_params { int nx, ny, ns, use_octree, spl, arith, seed_mode, max_depth, i0, i1, istep, j0, j1, jstep, threads; };
struct hs_counters { uint64_t rays, sphere_tests, aabb_tests, paths; uint32_t max_depth; };

struct HostTree {
    std::vector<uint2> vox;
    std::vector<uint32_t> refs, big_refs, prolog, ent_off;
    std::vector<uint16_t> ent_cell;
    GridView grid;
    float planes[3][kPlanes];
    bool no_drops = true;
};

static void make_planes(float P[3][kPlanes]) {
    const float lo[3] = {-11.f, 0.f, -11.f}, hi[3] = {11.f, 2.f, 11.f};
    for (int a = 0; a < 3; a++) {
        P[a][0] = lo[a]; P[a][8] = hi[a];
        for (int step = 8; step > 1; step >>= 1)
            for (int i = 0; i < 8; i += step) P[a][i + step / 2] = P[a][i] + (P[a][i + step] - P[a][i]) / 2;
    }
}

// voxel shape of slab-shaped scenes: the product's defaults; profiles/warp_model.py moves them (hs_set_grid_shape)
static float g_grid_flat = kGridFlat, g_grid_wide = kGridWide, g_pad_reach = kSceneReach;

// k_grid_prep + k_vox_pass: the big spheres (ascending index, up to kMaxBig) and the surface x voxel lists of the others, over
// the defined spheres i >= 1 that `take(i)`.  A hollow sphere (r < 0) is hit where |r| puts its surface: gridded by |r|.
template <typename Take>
static void build_grid(const std::vector<float4> &geom, const std::vector<int> &tag, Take take, float density, HostTree &T) {
    const int n = (int)geom.size();
    const float big_r = kBigRadiusFrac * 2.75f;
    std::vector<uint32_t> small;
    float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f};
    for (int i = 1; i < n; i++) {
        if (tag[(size_t)i] < 0 || !take(i)) continue;
        const float4 s = geom[(size_t)i];
        const float ar = fabsf(s.w);
        if (ar > big_r && (int)T.big_refs.size() < kMaxBig) { T.big_refs.push_back((uint32_t)i); continue; }
        small.push_back((uint32_t)i);
        const float r = ar + sphere_pad(ar, g_pad_reach);
        lo[0] = fminf(lo[0], s.x - r); hi[0] = fmaxf(hi[0], s.x + r);
        lo[1] = fminf(lo[1], s.y - r); hi[1] = fmaxf(hi[1], s.y + r);
        lo[2] = fminf(lo[2], s.z - r); hi[2] = fmaxf(hi[2], s.z + r);
    }
    memset(&T.grid, 0, sizeof T.grid);
    const uint32_t voxels = choose_grid(lo, hi, (uint32_t)small.size(), density, T.grid, g_grid_flat, g_grid_wide);
    if (voxels) {
        std::vector<std::vector<uint32_t>> lists(voxels);
        for (uint32_t idx : small) {
            float4 s = geom[idx];
            s.w = fabsf(s.w);
            const float pad = sphere_pad(s.w, g_pad_reach);
            int v0[3], v1[3];
            voxel_range(T.grid, s, pad, v0, v1);
            for (int z = v0[2]; z <= v1[2]; z++)
                for (int y = v0[1]; y <= v1[1]; y++)
                    for (int x = v0[0]; x <= v1[0]; x++) {
                        float blo[3], bhi[3];
                        voxel_box(T.grid, x, y, z, blo, bhi);
                        if (shell_hits_box(s, pad, blo, bhi)) lists[((size_t)z * T.grid.ny + y) * T.grid.nx + x].push_back(idx);
                    }
        }
        T.vox.resize(voxels);
        for (uint32_t v = 0; v < voxels; v++) {
            std::sort(lists[v].begin(), lists[v].end());
            T.vox[v].x = (uint32_t)T.refs.size();
            T.vox[v].y = (uint32_t)lists[v].size();
            T.refs.insert(T.refs.end(), lists[v].begin(), lists[v].end());
        }
    }
}

// Rebuild the traversal structure on the host from a reference-layout Octree blob: the per-sphere lists of cells that
// STORE the sphere come straight from the reference's leaf buckets.
static void build_host_tree(const std::vector<float4> &geom, const std::vector<int> &tag, const int32_t *blob, int spl,
                            float density, HostTree &T) {
    make_planes(T.planes);
    const int n = (int)geom.size();
    const int32_t *bn = blob;
    const int32_t *bl = blob + kNumberNodes * kNodeInts;
    const int32_t *cnt = bl + (size_t)(kNumberLeafs + 1) * (size_t)(spl + 1);
    const int node_count = cnt[0];
    auto plane_index = [&](int a, float v) { for (int i = 0; i < kPlanes; i++) if (T.planes[a][i] == v) return i; return -1; };
    std::vector<std::vector<uint16_t>> cells_of((size_t)n);
    for (int ni = 0; ni < node_count; ni++) {
        const int32_t *nd = bn + ni * kNodeInts;
        if (nd[0] != 3) continue;
        const float *bx = reinterpret_cast<const float *>(nd + 1);
        const int m = morton_of(plane_index(0, bx[0]), plane_index(1, bx[1]), plane_index(2, bx[2]));
        for (int c = 0; c < 8; c++) {
            const int leaf = nd[7 + c];
            if (leaf == 0) break;
            const int32_t *lf = bl + (size_t)leaf * (size_t)(spl + 1);
            for (int j = 0; j < lf[spl]; j++) cells_of[(size_t)lf[j]].push_back((uint16_t)m);
        }
    }
    // did the reference drop an entry?  (a defined sphere `intersects` more level-3 boxes than leaf buckets list it in;
    // acceleration_structure.h:82-93 with its float expansion and the (low, high] x interval)
    T.no_drops = true;
    for (int i = 1; i < n && T.no_drops; i++) {
        const float4 s = geom[(size_t)i];
        int cnt[3] = {0, 0, 0};
        for (int a = 0; a < 3; a++) {
            const float c = a == 0 ? s.x : (a == 1 ? s.y : s.z);
            for (int k = 0; k < 8; k++) {
                const float lo = T.planes[a][k] - s.w, hi = T.planes[a][k + 1] + s.w;
                cnt[a] += (a == 0 ? c > lo : c >= lo) && c <= hi;
            }
        }
        if ((size_t)(cnt[0] * cnt[1] * cnt[2]) != cells_of[(size_t)i].size()) T.no_drops = false;
    }
    T.ent_off.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++) {
        T.ent_off[(size_t)i] = (uint32_t)T.ent_cell.size();
        T.ent_cell.insert(T.ent_cell.end(), cells_of[(size_t)i].begin(), cells_of[(size_t)i].end());
    }
    T.ent_off[(size_t)n] = (uint32_t)T.ent_cell.size();
    build_grid(geom, tag, [&](int i) { return !cells_of[(size_t)i].empty(); }, density, T);
}

// The flat-list mode's grid (OctreeBuilder::build with all_spheres): every defined sphere but slot 0, wherever it lies.
static void build_list_grid(const std::vector<float4> &geom, const std::vector<int> &tag, float density, HostTree &T) {
    make_planes(T.planes);
    T.ent_off.assign(geom.size() + 1, 0u);
    build_grid(geom, tag, [](int) { return true; }, density, T);
}

static void view_of(HostTree &T, TreeView &tv, bool slot0_none, bool check_visibility = true) {
    T.prolog.assign(1, 0u);
    T.prolog.insert(T.prolog.end(), T.big_refs.begin(), T.big_refs.end());
    memset(&tv, 0, sizeof tv);
    tv.grid = T.grid;
    tv.grid.vox = T.vox.data(); tv.grid.refs = T.refs.data();
    tv.vis.ent_off = T.ent_off.data(); tv.vis.ent_cell = T.ent_cell.data();
    tv.prolog = T.prolog.data(); tv.nprolog = (int)T.prolog.size();
    tv.check_visibility = check_visibility ? 1 : 0;
    tv.slot0_none = slot0_none ? 1 : 0;
    memcpy(tv.planes, T.planes, sizeof tv.planes);
    tv.no_drops = T.no_drops ? 1 : 0;
    for (int a = 0; a < 3; a++) tv.cell_inv[a] = 8.0f / (T.planes[a][kPlanes - 1] - T.planes[a][0]);
}

// ---- host emulation of k_render_coop's candidate rule (rt_coop.cuh coop_trace), one ray at a time -------------------------
// What the cooperative kernel does differently from trace_walk: candidates only pass the conservative pre-filter
// (maybe_hit_ub) against  min(pruning bound, exit of the ray's current voxel + slack)  — a root beyond the voxel is left to the
// voxel that holds it — certain hits lower the pruning bound before they are evaluated, and the exact tests run later, in any
// order.  `eager`: the queued candidates are evaluated after every voxel (the bound follows the exact values at once);
// otherwise only at the end of the trace (the walk is steered by the certain-hit bounds alone).  Both extremes — and every
// schedule between them, which is what the warp's ring does — must return trace_walk's minimum.
static const float kCoopExitSlackRel = 1e-4f, kCoopExitSlackAbs = 1e-4f;      // rt_coop.cuh kVoxelExitSlack*
struct CoopHit { float t; int idx; bool tie; };
static CoopHit coop_walk_host(const SceneView &sc, const TreeView &tv, const vec3f o, const vec3f d, const bool eager) {
    const float a = dot3(d, d), ia = rcp_trav(a);
    CoopHit h;
    h.t = kTMax; h.idx = -1; h.tie = false;
    float bound = kTMax;
    std::vector<int> ring;
    auto drain = [&]() {
        for (int idx : ring) {
            float t;
            if (sphere_test(sc.geom[idx], o, d, a, kTMax, t)) {
                if (t < h.t) { h.t = t; h.idx = idx; h.tie = false; }
                else if (t == h.t && idx != h.idx) h.tie = true;
            }
        }
        ring.clear();
        bound = fminf(bound, h.t);
    };
    { float t; if (!tv.slot0_none && sphere_test(sc.geom[0], o, d, a, kTMax, t)) { h.t = t; h.idx = 0; bound = t; } }
    for (int k = 1; k < tv.nprolog; k++) {
        const int idx = (int)tv.prolog[k];
        float ub;
        if (maybe_hit_ub(sc.geom[idx], o, d, a, ia, bound, ub)) { if (ub < bound) bound = ub; ring.push_back(idx); }
    }
    const GridView &g = tv.grid;
    RayPre r;
    r.o = o; r.d = d; r.a = a;
    r.inv = mk(rcp_trav(d.x), rcp_trav(d.y), rcp_trav(d.z));
    float te, t_exit;
    if (g.nx != 0 && ray_box(r, g.org, g.hi, bound * (1.0f + kTSlackRel) + kTSlackAbs, te, t_exit)) {
        int ix = (int)floorf((o.x + d.x * te - g.org[0]) * g.inv_vs[0]);
        int iy = (int)floorf((o.y + d.y * te - g.org[1]) * g.inv_vs[1]);
        int iz = (int)floorf((o.z + d.z * te - g.org[2]) * g.inv_vs[2]);
        ix = imin(imax(ix, 0), g.nx - 1); iy = imin(imax(iy, 0), g.ny - 1); iz = imin(imax(iz, 0), g.nz - 1);
        const int sx = d.x >= 0.0f ? 1 : -1, sy = d.y >= 0.0f ? 1 : -1, sz = d.z >= 0.0f ? 1 : -1;
        float tmx = fabsf(d.x) >= kDdaMinDir ? (g.org[0] + (float)(ix + (sx > 0)) * g.vs[0] - o.x) * r.inv.x : kTMax;
        float tmy = fabsf(d.y) >= kDdaMinDir ? (g.org[1] + (float)(iy + (sy > 0)) * g.vs[1] - o.y) * r.inv.y : kTMax;
        float tmz = fabsf(d.z) >= kDdaMinDir ? (g.org[2] + (float)(iz + (sz > 0)) * g.vs[2] - o.z) * r.inv.z : kTMax;
        const float dtx = fabsf(g.vs[0] * r.inv.x), dty = fabsf(g.vs[1] * r.inv.y), dtz = fabsf(g.vs[2] * r.inv.z);
        int budget = g.nx + g.ny + g.nz + 4;
        bool walking = true;
        while (walking) {
            const uint2 v = g.vox[((size_t)(iz * g.ny + iy) * g.nx + ix)];
            if (v.y) {
                const float t_out = fminf(tmx, fminf(tmy, tmz)) * (1.0f + kCoopExitSlackRel) + kCoopExitSlackAbs;
                const float round_bound = bound;          // the chunks of one round may all see the bound the round began with
                for (uint32_t k = v.x; k < v.x + v.y; k++) {
                    const int idx = (int)g.refs[k];
                    float ub;
                    if (maybe_hit_ub(sc.geom[idx], o, d, a, ia, fminf(eager ? bound : round_bound, t_out), ub)) {
                        if (ub < bound) bound = ub;
                        ring.push_back(idx);
                    }
                }
                if (eager) drain();
            }
            float t_in;
            if (tmx <= tmy && tmx <= tmz) { t_in = tmx; ix += sx; tmx += dtx; walking = (unsigned)ix < (unsigned)g.nx; }
            else if (tmy <= tmz)          { t_in = tmy; iy += sy; tmy += dty; walking = (unsigned)iy < (unsigned)g.ny; }
            else                          { t_in = tmz; iz += sz; tmz += dtz; walking = (unsigned)iz < (unsigned)g.nz; }
            if (t_in > bound * (1.0f + kTSlackRel) + kTSlackAbs || t_in > t_exit * (1.0f + 1e-5f) + 1e-6f || --budget < 0) walking = false;
        }
    }
    drain();
    return h;
}
static bool g_coop_check = false, g_list_grid = false;
static unsigned long long g_coop_rays = 0, g_coop_bad = 0;

extern "C" {

void hs_set_grid_shape(float flat, float wide) { g_grid_flat = flat; g_grid_wide = wide; }
void hs_set_pad_reach(float reach) { g_pad_reach = reach; }
// every octree (or list-grid) ray of the following renders is also traced by coop_walk_host (both schedules) and compared with trace_walk's minimum
// use_octree = 0 renders go through the flat-list mode's grid (hitable_list::hit answered by trace_tree without the visibility
// rule), as the library does from kListGridMinSpheres spheres on; off: the plain list sweep (trace_list)
void hs_set_list_grid(int on) { g_list_grid = on != 0; }
void hs_coop_check(int on) { g_coop_check = on != 0; g_coop_rays = g_coop_bad = 0; }
void hs_coop_check_result(unsigned long long *rays, unsigned long long *mismatches) { *rays = g_coop_rays; *mismatches = g_coop_bad; }
// choose_grid as the build calls it (the product's default voxel shape): dims[3]; returns the voxel count
unsigned hs_choose_grid(const float *lo, const float *hi, unsigned live, float density, int *dims) {
    GridView g;
    memset(&g, 0, sizeof g);
    const uint32_t v = choose_grid(lo, hi, live, density, g);
    dims[0] = g.nx; dims[1] = g.ny; dims[2] = g.nz;
    return v;
}

// camera22: origin, llc, horizontal, vertical, u, v, w, lens_radius (taken from the oracle so that only the
// hot path is under test here)
static int render_core(const hs_sphere *sph, int n, const float *camera22, const void *blob, const hs_params *p, float density,
              float *fb_gamma, float *fb_linear, hs_counters *ctr_out, uint64_t *build_stats /* voxels, refs */,
              const TreeView *given) {
    std::vector<float4> geom((size_t)n), matl((size_t)n);
    std::vector<int> tag((size_t)n);
    for (int i = 0; i < n; i++) {
        geom[(size_t)i] = make_float4(sph[i].cx, sph[i].cy, sph[i].cz, sph[i].radius);
        matl[(size_t)i] = make_float4(sph[i].ax, sph[i].ay, sph[i].az, sph[i].param);
        tag[(size_t)i] = sph[i].mat;
    }
    SceneView sc;
    sc.geom = geom.data(); sc.matl = matl.data(); sc.tag = tag.data(); sc.n = n;
    HostTree T;
    TreeView tv;
    memset(&tv, 0, sizeof tv);
    if (p->use_octree && given) {
        tv = *given;
        make_planes(T.planes);
        memcpy(tv.planes, T.planes, sizeof tv.planes);
        for (int a = 0; a < 3; a++) tv.cell_inv[a] = 8.0f / (T.planes[a][kPlanes - 1] - T.planes[a][0]);
    } else if (p->use_octree) {
        build_host_tree(geom, tag, static_cast<const int32_t *>(blob), p->spl, density, T);
        view_of(T, tv, tag[0] < 0);
        if (build_stats) { build_stats[0] = T.vox.size(); build_stats[1] = T.refs.size(); }
    } else if (g_list_grid) {
        build_list_grid(geom, tag, density, T);
        view_of(T, tv, tag[0] < 0, false);
        if (build_stats) { build_stats[0] = T.vox.size(); build_stats[1] = T.refs.size(); }
    }
    const bool tree = p->use_octree || g_list_grid;
    CameraData cam;
    memcpy(&cam, camera22, sizeof cam);
    hs_counters total;
    memset(&total, 0, sizeof total);
    const int nrows = (p->j1 - p->j0 + p->jstep - 1) / p->jstep;
#pragma omp parallel
    {
        hs_counters c;
        memset(&c, 0, sizeof c);
#pragma omp for schedule(dynamic, 1)
        for (int r = 0; r < nrows; r++) {
            const int j = p->j0 + r * p->jstep;
            for (int i = p->i0; i < p->i1; i += p->istep) {
                const int pix = j * p->nx + i;
                xorwow rng;
                xorwow_seed(rng, (unsigned long long)(long long)(1984 + pix));
                vec3f col = mk(0, 0, 0);
                for (int s = 0; s < p->ns; s++) {
                    const float u = div_(add_((float)i, xorwow_uniform(rng)), (float)p->nx);
                    const float v = div_(add_((float)j, xorwow_uniform(rng)), (float)p->ny);
                    vec3f o, d, att = mk(1, 1, 1), contrib = mk(0, 0, 0);
                    camera_ray(cam, u, v, rng, o, d);
                    c.paths++;
                    for (int depth = 0; depth < p->max_depth; depth++) {
                        c.rays++;
                        TraceCounters tcn{};
                        Hit h = tree ? trace_tree(sc, tv, &tv.planes[0][0], o, d, tcn)
                                     : trace_list(sc.geom, sc.tag, sc.n, o, d, tcn);
                        if (g_coop_check && tree) {
                            bool tie = false;
                            const Hit m = trace_walk<kWalkMin>(sc, tv, &tv.planes[0][0], o, d, tcn, 0.0f, &tie);
                            unsigned long long bad = 0;
                            for (int eager = 0; eager < 2; eager++) {
                                const CoopHit c2 = coop_walk_host(sc, tv, o, d, eager != 0);
                                bad += !(c2.t == m.t && c2.tie == tie && (tie || c2.idx == m.idx));
                            }
#pragma omp atomic
                            g_coop_rays += 1;
#pragma omp atomic
                            g_coop_bad += bad;
                        }
                        if (h.idx >= 0) {
                            vec3f hp, hn, a, dn;
                            hit_point(geom[(size_t)h.idx], o, d, h.t, hp, hn);
                            if (!scatter(tag[(size_t)h.idx], matl[(size_t)h.idx], d, hp, hn, a, dn, rng)) break;
                            att = mk(mul_(att.x, a.x), mul_(att.y, a.y), mul_(att.z, a.z));
                            o = hp; d = dn;
                        } else {
                            const vec3f k = sky(d);
                            contrib = mk(mul_(att.x, k.x), mul_(att.y, k.y), mul_(att.z, k.z));
                            break;
                        }
                    }
                    col = mk(add_(col.x, contrib.x), add_(col.y, contrib.y), add_(col.z, contrib.z));
                }
                if (fb_linear) { fb_linear[3 * (size_t)pix] = col.x; fb_linear[3 * (size_t)pix + 1] = col.y; fb_linear[3 * (size_t)pix + 2] = col.z; }
                if (fb_gamma) {
                    const float k = div_(1.0f, (float)p->ns);
                    fb_gamma[3 * (size_t)pix] = sqrt_(mul_(col.x, k));
                    fb_gamma[3 * (size_t)pix + 1] = sqrt_(mul_(col.y, k));
                    fb_gamma[3 * (size_t)pix + 2] = sqrt_(mul_(col.z, k));
                }
            }
        }
#pragma omp critical
        { total.rays += c.rays; total.paths += c.paths; }
    }
    if (ctr_out) *ctr_out = total;
    return 0;
}


int hs_render(const hs_sphere *sph, int n, const float *camera22, const void *blob, const hs_params *p, float density,
              float *fb_gamma, float *fb_linear, hs_counters *ctr_out, uint64_t *build_stats) {
    return render_core(sph, n, camera22, blob, p, density, fb_gamma, fb_linear, ctr_out, build_stats, nullptr);
}

// Same renderer over traversal arrays produced elsewhere (the GPU build, read back with rt_octree_debug_read):
// grid_desc = 12 floats (org, hi, vs, inv_vs) + 3 ints (nx, ny, nz).
int hs_render_with_tree(const hs_sphere *sph, int n, const float *camera22, const hs_params *p, float *fb_gamma,
                        hs_counters *ctr_out, const void *grid_desc, const void *vox, const void *refs,
                        const void *ent_off, const void *ent_cell, const void *big_refs, int nbig) {
    TreeView tv;
    memset(&tv, 0, sizeof tv);
    const float *gf = static_cast<const float *>(grid_desc);
    const int *gi = reinterpret_cast<const int *>(gf + 12);
    for (int k = 0; k < 3; k++) { tv.grid.org[k] = gf[k]; tv.grid.hi[k] = gf[3 + k]; tv.grid.vs[k] = gf[6 + k]; tv.grid.inv_vs[k] = gf[9 + k]; }
    tv.grid.nx = gi[0]; tv.grid.ny = gi[1]; tv.grid.nz = gi[2];
    tv.grid.vox = static_cast<const uint2 *>(vox); tv.grid.refs = static_cast<const uint32_t *>(refs);
    tv.vis.ent_off = static_cast<const uint32_t *>(ent_off); tv.vis.ent_cell = static_cast<const uint16_t *>(ent_cell);
    std::vector<uint32_t> prolog(1, 0u);
    prolog.insert(prolog.end(), static_cast<const uint32_t *>(big_refs), static_cast<const uint32_t *>(big_refs) + nbig);
    tv.prolog = prolog.data(); tv.nprolog = (int)prolog.size();
    tv.check_visibility = 1;
    tv.slot0_none = sph[0].mat < 0;
    tv.no_drops = 1;
    for (uint32_t k = 0, e = tv.vis.ent_off[n]; k < e; k++) if (tv.vis.ent_cell[k] & kEntDropped) tv.no_drops = 0;
    return render_core(sph, n, camera22, nullptr, p, 0.f, fb_gamma, nullptr, ctr_out, nullptr, &tv);
}

// The traversal structure of the scene: the octree's grid (use_octree, from the reference-layout blob) or the flat-list mode's grid
// over all spheres, and its view.
struct HostScene {
    std::vector<float4> geom;
    std::vector<int> tag;
    HostTree T;
    TreeView tv;
    SceneView sc;
};
static void host_scene(const hs_sphere *sph, int n, const void *blob, int spl, int use_octree, float density, HostScene &S) {
    S.geom.resize((size_t)n);
    S.tag.resize((size_t)n);
    for (int i = 0; i < n; i++) { S.geom[(size_t)i] = make_float4(sph[i].cx, sph[i].cy, sph[i].cz, sph[i].radius); S.tag[(size_t)i] = sph[i].mat; }
    if (use_octree) build_host_tree(S.geom, S.tag, static_cast<const int32_t *>(blob), spl, density, S.T);
    else build_list_grid(S.geom, S.tag, density, S.T);
    view_of(S.T, S.tv, S.tag[0] < 0, use_octree != 0);
    memset(&S.sc, 0, sizeof S.sc);
    S.sc.geom = S.geom.data(); S.sc.tag = S.tag.data(); S.sc.n = n;
}

// Closest hit of caller rays (3 floats each) by the product's walks compiled for the host, over the octree's grid (use_octree) or
// the flat-list mode's grid: walk 0 trace_tree (k_trace_rays), 1 / 2 the cooperative candidate rule (coop_walk_host, eager / lazy
// schedule) followed by finish_hit, as coop_trace_tree.  out_idx = -1 on a miss.
int hs_trace_rays(const hs_sphere *sph, int n, const void *blob, int spl, int use_octree, float density, int walk, int nrays,
                  const float *org, const float *dir, int *out_idx, float *out_t) {
    if (walk < 0 || walk > 2 || (use_octree && !blob) || n < 1) return -1;
    HostScene S;
    host_scene(sph, n, blob, spl, use_octree, density, S);
    const float *planes = &S.tv.planes[0][0];
#pragma omp parallel for schedule(dynamic, 64)
    for (int k = 0; k < nrays; k++) {
        const vec3f o = mk(org[3 * (size_t)k], org[3 * (size_t)k + 1], org[3 * (size_t)k + 2]);
        const vec3f d = mk(dir[3 * (size_t)k], dir[3 * (size_t)k + 1], dir[3 * (size_t)k + 2]);
        TraceCounters tc{};
        Hit h;
        if (walk == 0) {
            h = trace_tree(S.sc, S.tv, planes, o, d, tc);
        } else {
            const CoopHit c = coop_walk_host(S.sc, S.tv, o, d, walk == 1);
            h.t = c.t; h.idx = c.idx;
            h = finish_hit(S.sc, S.tv, planes, o, d, h, c.tie, tc);
        }
        out_idx[k] = h.idx;
        out_t[k] = h.t;
    }
    return 0;
}

// The voxel grid the build makes for the scene (as hs_trace_rays): out9 = origin, voxel size, far corner; dims = nx, ny, nz;
// counts = voxels, references (the library's coop_items rule reads their ratio).
int hs_grid_geometry(const hs_sphere *sph, int n, const void *blob, int spl, int use_octree, float density, float *out9, int *dims,
                     uint64_t *counts) {
    if ((use_octree && !blob) || n < 1) return -1;
    HostScene S;
    host_scene(sph, n, blob, spl, use_octree, density, S);
    const GridView &g = S.T.grid;
    for (int k = 0; k < 3; k++) { out9[k] = g.org[k]; out9[3 + k] = g.vs[k]; out9[6 + k] = g.hi[k]; }
    dims[0] = g.nx; dims[1] = g.ny; dims[2] = g.nz;
    counts[0] = S.T.vox.size(); counts[1] = S.T.refs.size();
    return 0;
}

// Soundness of visible_fast (rt_trace.cuh) against the rule it short-cuts: for `nrays` pseudo-random rays — aimed at sphere
// surfaces, many of them with origins ON cell planes, axis-parallel or zero direction components, far-away origins and
// hits within 1e-3 of a cell face — every accepted root of every probed sphere is classified both ways.
// out[0] hits probed, out[1] fast accepts, out[2] exact accepts, out[3] fast accepts the exact rule REJECTS (must be 0).
int hs_visible_soundness(const hs_sphere *sph, int n, const void *blob, int spl, uint64_t seed, int nrays, uint64_t *out) {
    std::vector<float4> geom((size_t)n);
    std::vector<int> tag((size_t)n);
    for (int i = 0; i < n; i++) { geom[(size_t)i] = make_float4(sph[i].cx, sph[i].cy, sph[i].cz, sph[i].radius); tag[(size_t)i] = sph[i].mat; }
    HostTree T;
    TreeView tv;
    build_host_tree(geom, tag, static_cast<const int32_t *>(blob), spl, 4.0f, T);
    view_of(T, tv, tag[0] < 0);
    const float *planes = &tv.planes[0][0];
    uint64_t st = seed * 6364136223846793005ull + 1442695040888963407ull;
    auto rnd = [&]() { st = st * 6364136223846793005ull + 1442695040888963407ull; return (float)((st >> 40) & 0xffffff) / 16777216.0f; };
    out[0] = out[1] = out[2] = out[3] = 0;
    TraceCounters tc;
    tc.sphere_tests = tc.node_tests = tc.voxel_steps = 0;
    for (int r = 0; r < nrays; r++) {
        const int idx = 1 + (int)(rnd() * (float)(n - 1)) % (n - 1);
        const float4 s = geom[(size_t)idx];
        if (tag[(size_t)idx] < 0) continue;
        // a point on (or, for grazing rays, just outside) the sphere, and an origin somewhere around the scene
        float u = 2.f * rnd() - 1.f, ph = 6.2831853f * rnd(), q = sqrtf(fmaxf(0.f, 1.f - u * u));
        const float graze = (r % 7 == 0) ? 1.0f + 1e-4f * rnd() : 1.0f;
        vec3f target = mk(s.x + graze * s.w * q * cosf(ph), s.y + graze * s.w * u, s.z + graze * s.w * q * sinf(ph));
        vec3f o = mk(-14.f + 28.f * rnd(), -0.5f + 4.f * rnd(), -14.f + 28.f * rnd());
        const int kind = r % 11;
        if (kind == 1) o.x = planes[(int)(rnd() * 8.99f)];                          // origin exactly on a cell plane
        if (kind == 2) o.y = planes[kPlanes + (int)(rnd() * 8.99f)];
        if (kind == 3) o.z = planes[2 * kPlanes + (int)(rnd() * 8.99f)];
        if (kind == 4) o = mk(1e4f * (rnd() - 0.5f), 50.f * rnd(), 1e4f * (rnd() - 0.5f));   // far away
        if (kind == 5) {                                                            // target within 1e-3 of a cell face
            const int a = (int)(rnd() * 2.99f);
            const float pl = planes[a * kPlanes + (int)(rnd() * 8.99f)] + 2e-3f * (rnd() - 0.5f);
            if (a == 0) target.x = pl; else if (a == 1) target.y = pl; else target.z = pl;
        }
        vec3f d = mk(target.x - o.x, target.y - o.y, target.z - o.z);
        if (kind == 6) { o.x = target.x; d.x = 0.0f; }                              // zero direction components
        if (kind == 7) { o.z = target.z; d.z = -0.0f; }
        if (kind == 8) { o.x = target.x; o.z = target.z; d.x = 0.0f; d.z = 0.0f; }  // vertical ray
        if (kind == 9) d = mk(d.x * 1e-3f, d.y * 1e-3f, d.z * 1e-3f);              // short direction: large t
        const float a = dot3(d, d);
        // probe the aimed sphere and a few neighbours in index order (overlapping spheres in dense scenes)
        for (int dj = 0; dj < 4; dj++) {
            const int j = 1 + (idx - 1 + dj * 37) % (n - 1);
            if (tag[(size_t)j] < 0) continue;
            float t;
            if (!sphere_test(geom[(size_t)j], o, d, a, kTMax, t)) continue;
            int last_ok = -1;
            const bool fast = visible_fast(tv, planes, geom[(size_t)j], o, d, t);
            const bool exact = sphere_visible(tv.vis, planes, j, o, d, last_ok, tc);
            out[0]++; out[1] += fast; out[2] += exact; out[3] += fast && !exact;
        }
    }
    return 0;
}

}  // extern "C"
