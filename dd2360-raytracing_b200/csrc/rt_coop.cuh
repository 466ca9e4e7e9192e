// rt_coop.cuh — warp-cooperative closest hit ("flattened candidates") and the render kernel built on it.
// Included by rt_render.cu inside namespace rt.
//
// Why: in the pixel-per-lane walk (k_render) every lane tests the candidates of ITS OWN ray, so a warp runs as long as the
// lane with the longest candidate lists: profiles/warp_model.py (the product's traversal code replayed on the host in
// lock-step) shows, for BASELINE config 3, 28 % of the rays missing the grid altogether, 1.5 voxels visited per ray with
// ~13 references each, 0..75 candidates per ray — and 44 % of the lane-trips of the walk loop doing work.  The exact
// root evaluation (IEEE sqrt + two divisions) sat in that loop under a branch taken by 3.6 lanes.
//
// Here the lanes still own one pixel chain each (ray, RNG and pixel state in registers: rt_chain.cuh), but the
// candidate tests of the warp's 32 rays are pooled:
//   round   : every walking lane publishes the reference range of its CURRENT voxel; an inclusive warp scan lays the
//             ranges end to end (a flat list of `total` items of ITEMS consecutive references of one ray);
//   chunks  : 32 items at a time; item -> owner lane by a REDUX.OR of the segment ends + one POPC into a table of the lanes
//             that have items; the lane reads the owner's ray and pruning bound from shared memory, ITEMS float4 of list-order
//             geometry from L1/L2 and runs the conservative root pre-filter (maybe_hit_ub) on them.  The trip count is
//             warp-uniform (total / 32): no lane idles because its own ray had a short list;
//   bounds  : when the pre-filter makes a hit CERTAIN it also bounds the accepted root from above; a native shared-memory
//             atomicMin on the float's bits lowers the owner's pruning bound at once, so the walk and the later pre-filters
//             prune as sharply as with exact values while the exact evaluation waits;
//   ring    : candidates that pass (1.3 per ray at config 3) are appended to a per-warp ring in shared memory by ballot/popc
//             (no atomics: the warp is converged); whenever 32 are queued — and at the end of the trace — the lanes evaluate
//             the EXACT reference test (sphere.h:17-46, IEEE) on one entry each and fold (t, sphere index) into the owner's
//             record with two native 32-bit shared-memory atomics;
//   advance : owners re-read their bound and step the 3D-DDA to their next non-empty voxel (or stop).
// The closest hit of hitable_list::hit / hitTree is a strict-'<' minimum over a candidate set, so it does not depend on the
// order of evaluation (SURVEY D10); a candidate's accepted root does not depend on closest_so_far either:
//   sphere::hit(t_max) accepts root1 if t_min < root1 < t_max, else root2 if t_min < root2 < t_max; root2 >= root1 (the
//   rounding of (-b -+ sq)/a is monotone, a > 0), hence  hit(t_max) = [acc < t_max] with acc = root1 if root1 > t_min,
//   else root2 if root2 > t_min — exactly what sphere_test(.., t_max = FLT_MAX, ..) returns.
// Ties (two DIFFERENT spheres with bit-identical t) are detected here and ranked in the reference's test order by finish_hit.
#pragma once

namespace coop {

constexpr unsigned kFull = 0xffffffffu;
constexpr uint32_t kPrologFlag = 0x80000000u;    // ring reference: index into the prolog list instead of the voxel lists
constexpr int kRing = 160;
constexpr float kVoxelExitSlackRel = 1e-4f, kVoxelExitSlackAbs = 1e-4f;   // covers the DDA's accumulated rounding (<= ~700 additions per axis)                       // >= 31 (left over) + 128 (one chunk's pushes at four candidates per lane)

struct __align__(16) RayMeta {
    int koff;        // first reference of the lane's current voxel - ITEMS * its offset in the flat item list
    int kend;        // one past the last reference of that voxel
    float bound;     // what the pre-filter and the walk prune against: an upper bound of the ray's closest hit — the exact t of
                     // best_t, or less: the certain-hit bound of a candidate still waiting in the ring (maybe_hit_ub)
    float t_out;     // where the ray leaves its current voxel (+ slack): a root beyond it belongs to a later voxel, which lists the
                     // sphere too (the lists cover the padded surface) and offers it when the walk gets there — so a sphere that spans
                     // several voxels of the ray is queued for its exact test once, not once per voxel
};

struct __align__(16) WarpShared {
    float4 ro[32];                   // ray origin, a = dot(d, d)
    float4 rd[32];                   // ray direction, 1/a (approximate: pre-filter only)
    RayMeta meta[32];
    uint32_t best_t[32];             // closest hit so far: float bits of t (positive floats order like their bits) ...
    uint32_t best_i[32];             // ... and its sphere index (0xffffffff: none); provisional among equal t (the smallest seen)
    uint32_t tie[32];                // 1: two DIFFERENT spheres share best_t — finish_hit ranks them in the reference's order
    uint32_t slot[32];               // the lanes that have items this round, in lane order (item -> owner lookup)
    uint2 ring[kRing];               // {owner lane, reference}
};

// Exact test of up to 32 queued candidates, one per lane, folded into the owners' (t, index) records: minimum t, and among
// bit-identical t the smallest sphere index.  Two native 32-bit shared-memory atomics (ATOMS.MIN) instead of one 64-bit
// atomicMin, which is a compare-and-swap loop in shared memory (7.6 % of the stall samples of the first version of this
// kernel, profiles r02c); MATCH.ANY + REDUX per owner group was tried and is far slower (it serialises over the distinct
// owners: 34.0 instead of 21.9 ms per 8-spp frame).  Every lane is also the OWNER of ray `lane`: between the two atomics it resets the
// index of its own record if this drain lowered its t.  Entries [first, first + n).  Returns the owner's new t.
__device__ __forceinline__ float drain(WarpShared &ws, const SceneView &sc, const TreeView &tv, const unsigned lane, const int first, const int n) {
    const uint32_t before = ws.best_t[lane];
    __syncwarp();                                               // (no lane's atomic may overtake another lane's read of `before`)
    uint32_t owner = 0, tb = 0xffffffffu, idx = 0xffffffffu;
    if ((int)lane < n) {
        const uint2 e = ws.ring[first + (int)lane];
        const float4 ro = ws.ro[e.x], rd = ws.rd[e.x];
        const bool pro = (e.y & kPrologFlag) != 0u;
        const uint32_t k = e.y & ~kPrologFlag;
        const float4 s = pro ? __ldg(tv.prolog_geom + k) : __ldg(tv.grid.ref_geom + k);
        float t;
        if (sphere_test(s, mk(ro.x, ro.y, ro.z), mk(rd.x, rd.y, rd.z), ro.w, kTMax, t)) {
            idx = pro ? __ldg(tv.prolog + k) : __ldg(tv.grid.refs + k);
            tb = __float_as_uint(t);
            owner = e.x;
            atomicMin(&ws.best_t[owner], tb);
        }
    }
    __syncwarp();
    const uint32_t now = ws.best_t[lane];
    if (now != before) {                                        // a closer hit: whatever was recorded belongs to the old t
        ws.best_i[lane] = 0xffffffffu;
        ws.tie[lane] = 0u;
    }
    __syncwarp();
    if (tb != 0xffffffffu && ws.best_t[owner] == tb) {
        const uint32_t old = atomicMin(&ws.best_i[owner], idx);
        if (old != 0xffffffffu && old != idx) ws.tie[owner] = 1u;       // same root, another sphere (rt_trace.cuh "Ties")
    }
    ws.meta[lane].bound = fminf(ws.meta[lane].bound, __uint_as_float(now));     // (the bound may already be lower: certain hits not drained yet)
    __syncwarp();
    return __uint_as_float(now);
}

// Append the candidates flagged in `pass` (bit j: reference ref + j passed the pre-filter; N candidates per lane) to the ring by
// ballot/popc ranking — the warp is converged, `count` is a warp-uniform register, no atomics; drains while 32 or more are
// queued.  (Claiming slots with a shared-memory atomicAdd under the lanes' own predicates measured 3 % slower, profiles r02k.)
template <int N>
__device__ __forceinline__ void push_n(WarpShared &ws, const SceneView &sc, const TreeView &tv, const unsigned lane, const uint32_t pass,
                                       const uint32_t owner, const uint32_t ref, int &count) {
    unsigned m[N];
    unsigned any = 0u;
#pragma unroll
    for (int j = 0; j < N; j++) {
        m[j] = __ballot_sync(kFull, (pass >> j) & 1u);
        any |= m[j];
    }
    if (!any) return;
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll
    for (int j = 0; j < N; j++) {
        if ((pass >> j) & 1u) ws.ring[count + __popc(m[j] & lt)] = make_uint2(owner, ref + (uint32_t)j);
        count += __popc(m[j]);
    }
    __syncwarp();
    while (count >= 32) {
        drain(ws, sc, tv, lane, count - 32, 32);      // the newest 32; what is left stays at the front
        count -= 32;
    }
}

// Closest hit for the rays of the whole warp (lane `has` a ray or idles along).  Every lane of the warp must call.
// ITEMS = candidates per lane and chunk step (1, 2 or 4: a lane takes that many consecutive references of one voxel list, so the
// owner lookup and the ray fetch are paid once per group and the geometry loads are in flight together; 2 is the default,
// 4 pays off once lists are long — BASELINE config 5 has 71 references per voxel).
// Returns the minimum over ALL candidates and whether two different spheres tied for it (finish_hit settles ties and the
// visibility rule, as in trace_tree).
template <int ITEMS>
__device__ __forceinline__ Hit coop_trace(WarpShared &ws, const SceneView &sc, const TreeView &tv, const unsigned lane, const bool has,
                                          const vec3f o, const vec3f d, TraceCounters &tc, bool &tie) {
    const float a = dot3(d, d);
    const float ia = rcp_trav(a);
    __syncwarp();
    ws.ro[lane] = make_float4(o.x, o.y, o.z, a);
    ws.rd[lane] = make_float4(d.x, d.y, d.z, ia);
    ws.slot[lane] = lane;                   // (entries past this round's owners are read by lanes without an item: keep them lane ids)
    float best_t = kTMax;
    {   // ground sphere first, unconditionally (acceleration_structure.h:322-332) — unless slot 0 is undefined (never hit)
        uint32_t idx = 0xffffffffu;
        float t;
        if (has && !tv.slot0_none) {
            RT_COUNT(sphere_tests);
            if (sphere_test(__ldg(sc.geom), o, d, a, kTMax, t)) { best_t = t; idx = 0u; }
        }
        ws.best_t[lane] = __float_as_uint(best_t);
        ws.best_i[lane] = idx;
        ws.tie[lane] = 0u;
        ws.meta[lane].bound = best_t;
    }
    __syncwarp();
    int count = 0;
    for (int k = 1; k < tv.nprolog; k++) {   // big spheres: one pre-filter per lane, exact tests through the ring
        const float4 s = __ldg(tv.prolog_geom + k);
        if (has) RT_COUNT(sphere_tests);
        // most warps look nowhere near a given big sphere: the discriminant alone (the exact test's own float operations, so its
        // sign is the exact test's) settles that for the whole warp in a dozen instructions
        const vec3f oc = mk(sub_(o.x, s.x), sub_(o.y, s.y), sub_(o.z, s.z));
        const float bq = dot3(oc, d);
        const float disc = fma_(bq, bq, -mul_(a, fma_(-s.w, s.w, dot3(oc, oc))));
        if (!__any_sync(kFull, has && disc > 0.0f)) continue;
        float ub;
        const bool pass = has && maybe_hit_ub(s, o, d, a, ia, ws.meta[lane].bound, ub);
        if (pass && ub < ws.meta[lane].bound) ws.meta[lane].bound = ub;        // (the lane's own record: no other lane touches it here)
        push_n<1>(ws, sc, tv, lane, pass ? 1u : 0u, lane, kPrologFlag | (uint32_t)k, count);
    }
    best_t = ws.meta[lane].bound;           // from here on `best_t` is the pruning bound; exact values live in ws.best_t / best_i

    // ---- 3D-DDA set-up, per lane (as trace_walk) ----
    const GridView &g = tv.grid;
    bool walking = has && g.nx != 0;
    int ix = 0, iy = 0, iz = 0;
    float tmx = kTMax, tmy = kTMax, tmz = kTMax, dtx = 0.f, dty = 0.f, dtz = 0.f, t_exit = 0.f;
    const int sx = d.x >= 0.0f ? 1 : -1, sy = d.y >= 0.0f ? 1 : -1, sz = d.z >= 0.0f ? 1 : -1;
    uint32_t k = 0, cnt = 0;
    if (walking) {
        RayPre r;
        r.o = o; r.d = d; r.a = a;
        r.inv = mk(rcp_trav(d.x), rcp_trav(d.y), rcp_trav(d.z));
        float te;
        walking = ray_box(r, g.org, g.hi, best_t * (1.0f + kTSlackRel) + kTSlackAbs, te, t_exit);
        if (walking) {
            ix = (int)floorf((o.x + d.x * te - g.org[0]) * g.inv_vs[0]);
            iy = (int)floorf((o.y + d.y * te - g.org[1]) * g.inv_vs[1]);
            iz = (int)floorf((o.z + d.z * te - g.org[2]) * g.inv_vs[2]);
            ix = imin(imax(ix, 0), g.nx - 1);
            iy = imin(imax(iy, 0), g.ny - 1);
            iz = imin(imax(iz, 0), g.nz - 1);
            if (fabsf(d.x) > 0.0f) tmx = (g.org[0] + (float)(ix + (sx > 0)) * g.vs[0] - o.x) * r.inv.x;
            if (fabsf(d.y) > 0.0f) tmy = (g.org[1] + (float)(iy + (sy > 0)) * g.vs[1] - o.y) * r.inv.y;
            if (fabsf(d.z) > 0.0f) tmz = (g.org[2] + (float)(iz + (sz > 0)) * g.vs[2] - o.z) * r.inv.z;
            dtx = fabsf(g.vs[0] * r.inv.x); dty = fabsf(g.vs[1] * r.inv.y); dtz = fabsf(g.vs[2] * r.inv.z);
            RT_COUNT(voxel_steps);
            const uint2 v = __ldg(g.vox + ((size_t)(iz * g.ny + iy) * g.nx + ix));
            k = v.x; cnt = v.y;
        }
    }
    int budget = g.nx + g.ny + g.nz + 4;       // hard bound on voxel steps: the walk always terminates

    while (true) {
        // ---- advance the lanes whose voxel is empty (or used up) until every walking lane has candidates; each pass of
        //      this loop is one DDA step for the lanes that need it ----
        while (__any_sync(kFull, walking && cnt == 0u)) {
            if (walking && cnt == 0u) {
                float t_in;
                if (tmx <= tmy && tmx <= tmz) { t_in = tmx; ix += sx; tmx += dtx; walking = (unsigned)ix < (unsigned)g.nx; }
                else if (tmy <= tmz)          { t_in = tmy; iy += sy; tmy += dty; walking = (unsigned)iy < (unsigned)g.ny; }
                else                          { t_in = tmz; iz += sz; tmz += dtz; walking = (unsigned)iz < (unsigned)g.nz; }
                // a later voxel can only hold hits at t >= t_in (minus the float slack); also stop at the grid exit
                if (t_in > best_t * (1.0f + kTSlackRel) + kTSlackAbs || t_in > t_exit * (1.0f + 1e-5f) + 1e-6f || --budget < 0) walking = false;
                if (walking) {
                    RT_COUNT(voxel_steps);
                    const uint2 v = __ldg(g.vox + ((size_t)(iz * g.ny + iy) * g.nx + ix));
                    k = v.x; cnt = v.y;
                }
            }
        }
        if (!__any_sync(kFull, walking)) break;

        // ---- lay the lanes' reference ranges end to end, in units of ITEMS references ----
        const uint32_t mine = walking ? (cnt + (uint32_t)(ITEMS - 1)) / (uint32_t)ITEMS : 0u;
        uint32_t incl = mine;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, incl, off);
            if ((int)lane >= off) incl += v;
        }
        const uint32_t total = __shfl_sync(kFull, incl, 31);
        const uint32_t excl = incl - mine;
        ws.meta[lane].koff = (int)k - ITEMS * (int)excl;
        ws.meta[lane].kend = (int)(k + cnt);
        ws.meta[lane].t_out = fminf(tmx, fminf(tmy, tmz)) * (1.0f + kVoxelExitSlackRel) + kVoxelExitSlackAbs;
        // the lanes that have items, in lane order (= item order): slot[j] is the j-th of them
        const unsigned lt = (1u << lane) - 1u;
        const unsigned nz = __ballot_sync(kFull, mine > 0u);
        if (mine > 0u) ws.slot[__popc(nz & lt)] = lane;
        __syncwarp();

        uint32_t r0 = 0u;                       // rank in slot[] of the owner of item `base`
        for (uint32_t base = 0; base < total; base += 32u) {
            // a lane's last item is incl - 1: the segment ENDS inside this chunk are OR-reduced into one mask (REDUX); the owner of
            // item base + i is r0 + (ends before position i) lanes down the table; r0 moves on by the ends of the chunk
            const bool ends_here = mine > 0u && incl > base && incl <= base + 32u;
            const unsigned ends = __reduce_or_sync(kFull, ends_here ? 1u << (incl - 1u - base) : 0u);
            const uint32_t item = base + lane;
            const bool valid = item < total;
            const uint32_t owner = ws.slot[(r0 + (uint32_t)__popc(ends & lt)) & 31u];
            r0 += (uint32_t)__popc(ends);
            const float4 ro = ws.ro[owner], rd = ws.rd[owner];
            const RayMeta mt = ws.meta[owner];
            const uint32_t ref = (uint32_t)(mt.koff + ITEMS * (int)item);
            uint32_t pass = 0u;
            if (valid) {
                const vec3f oo = mk(ro.x, ro.y, ro.z), dd = mk(rd.x, rd.y, rd.z);
                float4 sg[ITEMS];
#pragma unroll
                for (int j = 0; j < ITEMS; j++) sg[j] = __ldg(g.ref_geom + ref + j);   // (past a list's end: the next list, or the slack elements)
                float ub = kTMax;
                const float t_far = fminf(mt.bound, mt.t_out);
#pragma unroll
                for (int j = 0; j < ITEMS; j++) {
                    float ubj;
                    RT_COUNT(sphere_tests);
                    const bool pj = maybe_hit_ub(sg[j], oo, dd, ro.w, rd.w, t_far, ubj) && (j == 0 || (int)ref + j < mt.kend);
                    if (pj) { pass |= 1u << j; ub = fminf(ub, ubj); }
                }
                // a certain hit lowers the owner's pruning bound at once (native shared-memory atomic on the float's bits: roots
                // are positive); its exact evaluation waits in the ring until 32 candidates are queued
                if (ub < mt.bound) atomicMin(reinterpret_cast<uint32_t *>(&ws.meta[owner].bound), __float_as_uint(ub));
            }
            push_n<ITEMS>(ws, sc, tv, lane, pass, owner, ref, count);
        }
        __syncwarp();
        best_t = ws.meta[lane].bound;           // no exact evaluation at the end of a round: the certain-hit bounds steer the walk
        cnt = 0u;                               // every published range was consumed: the advance loop steps on
    }
    while (count > 0) {                         // what is still queued: the last exact evaluations of this trace
        const int n = count < 32 ? count : 32;
        drain(ws, sc, tv, lane, count - n, n);
        count -= n;
    }
    Hit h;
    h.t = __uint_as_float(ws.best_t[lane]);
    h.idx = (int)ws.best_i[lane];               // 0xffffffff -> -1
    tie = ws.tie[lane] != 0u;
    return h;
}

// hitTree semantics on top of coop_trace: the visibility rule on the winner (as trace_tree), the rare failures re-walked per lane
template <int ITEMS>
__device__ __forceinline__ Hit coop_trace_tree(WarpShared &ws, const SceneView &sc, const TreeView &tv, const float *planes, const unsigned lane,
                                               const bool has, const vec3f o, const vec3f d, TraceCounters &tc) {
    bool tie = false;
    Hit h = coop_trace<ITEMS>(ws, sc, tv, lane, has, o, d, tc, tie);
    if (has) h = finish_hit(sc, tv, planes, o, d, h, tie, tc);
    return h;
}

// The lanes' pixel chains (rt_chain.cuh) are parked in shared memory during coop_trace (Chain::park) instead of being spilled to
// local memory by the register allocator; that is what lets 8 blocks per SM be resident (-9 % frame time over 6 blocks without
// parking, profiles r02r-r02t).  The body of k_render_coop and k_render_coop_pixels_progressive; MODE: rt_render.h LaunchMode.
template <int ITEMS, int MODE>
__device__ __forceinline__ void render_coop_lanes(const RenderLaunch &p) {
    __shared__ WarpShared wsh[kRenderThreads / 32];
    __shared__ uint32_t park[21][kRenderThreads];
    WarpShared &ws = wsh[threadIdx.x >> 5];
    const SceneView sc = p.scene;
    const unsigned lane = threadIdx.x & 31u;

    TraceCounters tc;
    tc.sphere_tests = tc.node_tests = tc.voxel_steps = 0;
    run_chains<MODE>(p, ChainF32(p), claim_batch(p), [&](Chain &c, const bool has) {
        c.park(park, threadIdx.x);
        __syncwarp();
        const Hit h = coop_trace_tree<ITEMS>(ws, sc, p.tree, &p.tree.planes[0][0], lane, has, c.o, c.d, tc);
        c.unpark(park, threadIdx.x);
        const float4 ro = ws.ro[lane], rd = ws.rd[lane];          // the ray itself is still where coop_trace published it
        c.o = mk(ro.x, ro.y, ro.z); c.d = mk(rd.x, rd.y, rd.z);
        return h;
    });
#ifdef RT_COUNTERS
    unsigned long long c64[3] = {tc.sphere_tests, tc.node_tests, tc.voxel_steps};
    for (int k = 0; k < 3; k++) {
        for (int off = 16; off > 0; off >>= 1) c64[k] += __shfl_xor_sync(kFull, c64[k], off);
        if (lane == 0) atomicAdd(p.counters + 2 + k, c64[k]);
    }
#endif
}
// LIST: pixel-list instances, as k_render's
template <int ITEMS, bool LIST = false>
__global__ void __launch_bounds__(kRenderThreads, 8) k_render_coop(const __grid_constant__ RenderLaunch p) {
    render_coop_lanes<ITEMS, LIST ? kModeList : kModeFrame>(p);
}
// progressive pixel lists, as k_render_pixels_progressive
template <int ITEMS>
__global__ void __launch_bounds__(kRenderThreads, 8) k_render_coop_pixels_progressive(const __grid_constant__ RenderLaunch p) {
    render_coop_lanes<ITEMS, kModeListProgressive>(p);
}

// test hook: closest hit of caller-supplied rays through the cooperative trace (32 rays per warp)
__global__ void __launch_bounds__(kRenderThreads) k_trace_rays_coop(const __grid_constant__ RenderLaunch p, const float *__restrict__ org,
                                                                   const float *__restrict__ dir, int n, int *__restrict__ out_idx,
                                                                   float *__restrict__ out_t) {
    __shared__ WarpShared wsh[kRenderThreads / 32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool has = i < n;
    const vec3f o = has ? mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]) : mk(0, 0, 0);
    const vec3f d = has ? mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]) : mk(0, 0, 1);
    TraceCounters tc;
    tc.sphere_tests = tc.node_tests = tc.voxel_steps = 0;
    const Hit h = coop_trace_tree<2>(wsh[threadIdx.x >> 5], p.scene, p.tree, &p.tree.planes[0][0], threadIdx.x & 31u, has, o, d, tc);
    if (has) { out_idx[i] = h.idx; out_t[i] = h.t; }
}

}  // namespace coop
