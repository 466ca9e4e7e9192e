// rt_render_half.cuh — the USE_FP16 render path (BASELINE config 4): render_init + render + color in half precision.
// (included by rt_render.cu; arithmetic in rt_half.cuh)
//
// Same persistent, queue-fed kernel shape as k_render (one pixel chain per lane, ballot/popc-compacted claims), with the
// per-lane state in half: ray, attenuation and — as in the reference, whose `vec3 col` is three halves (main.cu:101) —
// the pixel accumulator.  Octree mode walks the reference's own cells (rt_half.cuh coop_trace_h): the sub-grid of the
// FP32 path is built on float error bounds that half arithmetic does not honour.
#pragma once
// (rt_half.cuh is included by rt_render.cu at file scope)

namespace h16 {

// the FP16 create_world stores every centre, radius, albedo and parameter through real_t(float|double): the FP32 scene
// rounded once to half (main.cu:160-181).  8 bytes per sphere for geometry, 8 for the material.
__global__ void k_scene_to_half(const float4 *__restrict__ geom, const float4 *__restrict__ matl, int n, uint2 *__restrict__ geom_h,
                                uint2 *__restrict__ matl_h) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float4 g = geom[i], m = matl[i];
    __half2 a = __floats2half2_rn(g.x, g.y), b = __floats2half2_rn(g.z, g.w);
    geom_h[i] = make_uint2(*reinterpret_cast<uint32_t *>(&a), *reinterpret_cast<uint32_t *>(&b));
    a = __floats2half2_rn(m.x, m.y);
    b = __floats2half2_rn(m.z, m.w);
    matl_h[i] = make_uint2(*reinterpret_cast<uint32_t *>(&a), *reinterpret_cast<uint32_t *>(&b));
}

// Pair lists (rt_half.cuh PairView).  lists == 1: the flat mode, one list of all n spheres in index order;
// lists == kCells: the stored list of every level-3 cell (first cell_cap entries in ascending sphere order).
// Pass 1 (count) sizes the lists, a 513-thread scan makes the offsets, pass 2 writes the pairs.
__global__ void k_pairs_count(const int *__restrict__ tag, int n, int lists, const uint32_t *__restrict__ cell_start,
                              const uint32_t *__restrict__ cell_list, int cell_cap, uint32_t *__restrict__ pair_count) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= lists) return;
    uint32_t valid = 0;
    if (lists == 1) {
        for (int i = 0; i < n; i++) valid += tag[i] >= 0;
    } else {
        const uint32_t b = cell_start[m], e = min(cell_start[m + 1], b + (uint32_t)cell_cap);
        for (uint32_t k = b; k < e; k++) valid += tag[cell_list[k]] >= 0;
    }
    pair_count[m] = ((valid + 1u) / 2u + kPairPad - 1u) / kPairPad * kPairPad;       // padded with NaN pairs (coop_filter_h)
}
__global__ void k_pairs_scan(const uint32_t *__restrict__ pair_count, int lists, uint32_t *__restrict__ pair_start) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        uint32_t acc = 0;
        for (int m = 0; m < lists; m++) { pair_start[m] = acc; acc += pair_count[m]; }
        pair_start[lists] = acc;
    }
}
__global__ void k_pairs_fill(const uint2 *__restrict__ geom_h, const int *__restrict__ tag, int n, int lists,
                             const uint32_t *__restrict__ cell_start, const uint32_t *__restrict__ cell_list, int cell_cap,
                             const uint32_t *__restrict__ pair_start, uint4 *__restrict__ pair_geom, int2 *__restrict__ pair_idx) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= lists) return;
    uint32_t out = pair_start[m];
    int pend = -1;
    const unsigned short nan16 = 0x7e00u;
    auto emit = [&](int i0, int i1) {
        const uint2 g0 = geom_h[i0];
        uint2 g1 = make_uint2(0x7e007e00u, 0x7e007e00u);           // NaN sphere: the padding of an odd list
        if (i1 >= 0) g1 = geom_h[i1];
        (void)nan16;
        // g = {cx | cy << 16, cz | r << 16}; transpose to {cx0|cx1<<16, cy0|cy1<<16, cz0|cz1<<16, r0|r1<<16}
        pair_geom[out] = make_uint4((g0.x & 0xffffu) | (g1.x << 16), (g0.x >> 16) | (g1.x & 0xffff0000u),
                                    (g0.y & 0xffffu) | (g1.y << 16), (g0.y >> 16) | (g1.y & 0xffff0000u));
        pair_idx[out] = make_int2(i0, i1);
        out++;
    };
    auto feed = [&](int i) {
        if (tag[i] < 0) return;
        if (pend < 0) pend = i;
        else { emit(pend, i); pend = -1; }
    };
    if (lists == 1) {
        for (int i = 0; i < n; i++) feed(i);
    } else {
        const uint32_t b = cell_start[m], e = min(cell_start[m + 1], b + (uint32_t)cell_cap);
        for (uint32_t k = b; k < e; k++) feed((int)cell_list[k]);
    }
    if (pend >= 0) emit(pend, -1);
    for (const uint32_t end = pair_start[m + 1]; out < end; out++) {     // padding up to a multiple of kPairPad: NaN spheres, never hit
        pair_geom[out] = make_uint4(0x7e007e00u, 0x7e007e00u, 0x7e007e00u, 0x7e007e00u);
        pair_idx[out] = make_int2(-1, -1);
    }
}

// compact per-level tables of the octree nodes that exist (a node was created iff its subtree received an entry):
// ent[0..8) level 1, ent[8..72) level 2, ent[72..584) level 3; parents before children, each level in Morton order
__global__ void k_fp16_nodes(const uint32_t *__restrict__ cell_start, uint2 *__restrict__ ent, uint32_t *__restrict__ count) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    int pos1[8], pos2[64];
    uint32_t n1 = 0, n2 = 0, n3 = 0;
    for (int k = 0; k < 64 + 8; k++) count[4 + k] = 0u;
    for (int c1 = 0; c1 < 8; c1++) {
        pos1[c1] = -1;
        if (cell_start[c1 * 64 + 64] == cell_start[c1 * 64]) continue;
        pos1[c1] = (int)n1;
        ent[n1++] = make_uint2((uint32_t)(c1 >> 2) | (uint32_t)((c1 >> 1) & 1) << 8 | (uint32_t)(c1 & 1) << 16, 0u | (uint32_t)c1 << 16);
    }
    for (int m2 = 0; m2 < 64; m2++) {
        pos2[m2] = -1;
        if (cell_start[m2 * 8 + 8] == cell_start[m2 * 8]) continue;
        const int c1 = m2 >> 3, c2 = m2 & 7;
        const int x = (c1 >> 2) * 2 + (c2 >> 2), y = ((c1 >> 1) & 1) * 2 + ((c2 >> 1) & 1), z = (c1 & 1) * 2 + (c2 & 1);
        pos2[m2] = (int)n2;
        uint32_t &kid1 = count[4 + 64 + pos1[c1]];      // children of level-1 node pos1[c1] in the level-2 table: first | count << 16
        kid1 = (kid1 >> 16) ? kid1 + (1u << 16) : (n2 | 1u << 16);
        ent[8 + n2++] = make_uint2((uint32_t)x | (uint32_t)y << 8 | (uint32_t)z << 16, (uint32_t)pos1[c1] | (uint32_t)m2 << 16);
    }
    for (int m3 = 0; m3 < 512; m3++) {
        if (cell_start[m3 + 1] == cell_start[m3]) continue;
        int x, y, z;
        morton_to_xyz(m3, x, y, z);
        // count[4 + p]: the children of level-2 node p are contiguous in the level-3 table: first child | count << 16
        uint32_t &kid = count[4 + pos2[m3 >> 3]];
        kid = (kid >> 16) ? kid + (1u << 16) : (n3 | 1u << 16);
        ent[72 + n3++] = make_uint2((uint32_t)x | (uint32_t)y << 8 | (uint32_t)z << 16, (uint32_t)pos2[m3 >> 3] | (uint32_t)m3 << 16);
    }
    count[0] = n1; count[1] = n2; count[2] = n3;
}

// vec3.h:95-99 cross(): a*b - c*d -> fma(a,b,-(c*d)); the middle component's unary minus goes through float
__device__ __forceinline__ vec3h cross_h(const vec3h a, const vec3h b) {
    const hf cx = hfma_(vy(a), b.z, hneg_(hmul_(a.z, vy(b))));
    const hf cy = f2h(-h2f(hfma_(vx(a), b.z, hneg_(hmul_(a.z, vx(b))))));
    const hf cz = hfma_(vx(a), vy(b), hneg_(hmul_(vy(a), vx(b))));
    return mkh(cx, cy, cz);
}

// camera.h:22-44 under USE_FP16, evaluated on the device with the reference's own intrinsics (hsin / hcos / __hdiv);
// nvcc does not fold half intrinsics, so unlike the FP32 camera nothing here is a compile-time constant.
// out: 22 halves in CameraData order (origin, llc, horizontal, vertical, u, v, w, lens_radius).
__global__ void k_camera_setup_h(const float lfx, const float lfy, const float lfz, const float lax, const float lay, const float laz,
                                 const float upx, const float upy, const float upz, const float vfov_f, const int nx, const int ny,
                                 const float aspect_override, const float aperture_f, const float focus_f, __half *__restrict__ out) {
    const hf aperture = f2h(aperture_f), focus = f2h(focus_f), vfov = f2h(vfov_f);
    const hf aspect = aspect_override > 0.f ? f2h(aspect_override) : hdiv_(f2h((float)nx), f2h((float)ny));   // real_t(nx) / real_t(ny), main.cu:199
    const hf lens_radius = hdiv_(aperture, f2h(2.0f));
    const hf theta = hdiv_(hmul_(vfov, f2h(3.14159265358979323846f)), f2h(180.0f));
    const hf arg = hdiv_(theta, f2h(2.0f));
    const hf half_height = hdiv_(hsin(arg), hcos(arg));
    const hf half_width = hmul_(aspect, half_height);
    const vec3h lookfrom = mkh_f(lfx, lfy, lfz), lookat = mkh_f(lax, lay, laz), vup = mkh_f(upx, upy, upz);
    const vec3h w = unit_vectorh(vsub(lookfrom, lookat));
    const vec3h u = unit_vectorh(cross_h(vup, w));
    const vec3h v = cross_h(w, u);
    const hf hwf = hmul_(half_width, focus), hhf = hmul_(half_height, focus);
    const vec3h llc = vfma(w, hneg_(focus), vfma(v, hneg_(hhf), vfma(u, hneg_(hwf), lookfrom)));
    const vec3h horizontal = vscale(hmul_(hmul_(f2h(2.0f), half_width), focus), u);
    const vec3h vertical = vscale(hmul_(hmul_(f2h(2.0f), half_height), focus), v);
    const vec3h all[7] = {lookfrom, llc, horizontal, vertical, u, v, w};
    for (int k = 0; k < 7; k++) { out[3 * k] = vx(all[k]); out[3 * k + 1] = vy(all[k]); out[3 * k + 2] = all[k].z; }
    out[21] = lens_radius;
}

// PROG: progressive calls (p.accumulate, p.state_out) get instances of their own: compiled into the whole-frame instances, the
// two per-pixel branches cost 1.6 % of a C4 frame (2 602 vs 2 559 ms, B200 at 1000 W).
// LIST: pixel-list instances.  With PROG = false they are k_render's kModeList (`pix` is the lane's list slot); with PROG = true
// kModeListProgressive (`pix` is the frame pixel, whose sum continues in `out` and whose stream is resumed from and stored back
// to seed_states: the list pointer holds state_out's slot).
template <bool OCTREE, bool PROG, bool LIST = false>
__global__ void __launch_bounds__(kRenderThreads, 5)
k_render_h(const __grid_constant__ RenderLaunch p, const uint2 *__restrict__ geom_h, const uint2 *__restrict__ matl_h,
           const __half *__restrict__ cam_h, const PairView pv, const NodeTab nt) {
    __shared__ CoopSmem coop_sm[kRenderThreads / 32];
    __shared__ hf planes_h[3 * kPlanes];      // the slab planes of the octree boxes, rounded to half as AABB's real_t members are
    if (OCTREE && threadIdx.x < 3 * kPlanes) planes_h[threadIdx.x] = f2h((&p.tree.planes[0][0])[threadIdx.x]);
    __syncthreads();
    const CameraH cam = load_camera_h(cam_h);
    const unsigned lane = threadIdx.x & 31u;
    if (lane == 0) {
        coop_sm[threadIdx.x >> 5].tail = 0u;
        coop_sm[threadIdx.x >> 5].pairs_lo = coop_sm[threadIdx.x >> 5].pairs_hi = 0u;
    }
    __syncwarp();
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int pix = -1, pi = 0, pj = 0, s = 0, depth = 0;
    xorwow rng;
    rng.d = rng.v0 = rng.v1 = rng.v2 = rng.v3 = rng.v4 = 0;
    const hf zero = f2h(0.0f), one = f2h(1.0f);
    vec3h o = mkh(zero, zero, zero), d = mkh(zero, zero, one), att = mkh(one, one, one), col = mkh(zero, zero, zero);
    uint32_t nrays = 0, npaths = 0;
    bool exhausted = false;
    uint32_t stock_next = gwarp * 32u, stock_end = stock_next + 32u;
    const hf nxh = f2h((float)p.nx), nyh = f2h((float)p.ny);
    const hf inv_ns = inv_ns_h(p.ns_total);

    while (true) {
        while (true) {          // claim pixels for idle lanes (as k_render)
            const bool need = pix < 0 && !exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (!m) break;
            // single pixels from the frame-wide queue (batch 1): here the warp traces its lanes' rays one after the other, each a
            // scan of ~2 000 candidates, so balance between warps matters and the per-warp tile stock measured 3 - 14 % slower
            const uint32_t item = claim_items(p, m, lane, stock_next, stock_end, 1u);
            if (need) {
                if (item >= p.total_items) {
                    exhausted = true;
                } else if (LIST ? list_to_pixel(p, item, pi, pj, !PROG) : item_to_pixel(p, item, pi, pj)) {
                    pix = LIST && !PROG ? (int)item : pj * p.nx + pi;
                    s = 0; depth = 0;
                    col = mkh(zero, zero, zero);
                    if (PROG && p.accumulate) {  // progressive: the stored sums are halves widened to float, so this is exact
                        const float *acc = p.out + (size_t)pix * 3;
                        col = mkh_f(acc[0], acc[1], acc[2]);
                    }
                    pixel_stream(p, LIST && !p.seed_states ? pj * p.nx + pi : pix, rng);
                }
            }
        }
        if (!__ballot_sync(0xffffffffu, pix >= 0)) break;

        const bool have = pix >= 0;
        if (have) {
            if (depth == 0) {   // main.cu:104-106: real_t(i + U) / real_t(max_x) — the sum is float, the quotient __hdiv
                const hf u = hdiv_(f2h(__fadd_rn((float)pi, xorwow_uniform(rng))), nxh);
                const hf v = hdiv_(f2h(__fadd_rn((float)pj, xorwow_uniform(rng))), nyh);
                camera_ray_h(cam, u, v, rng, o, d);
                att = mkh(one, one, one);
                npaths++;
            }
            nrays++;
        }
        // closest hit of every lane's ray, one ray at a time by the whole warp (rt_half.cuh coop_trace_h)
        const HitH h = coop_trace_h<OCTREE>(coop_sm[threadIdx.x >> 5], planes_h, pv, nt, geom_h, have, o, d);
        if (have) {
            bool sample_done = false;
            vec3h contrib = mkh(zero, zero, zero);
            if (h.idx >= 0) {
                vec3h hp, hn, a, dn;
                hit_point_h(load_sphere_h(geom_h, h.idx), o, d, h.t, hp, hn);
                if (scatter_h(__ldg(p.scene.tag + h.idx), load_mat_h(matl_h, h.idx), d, hp, hn, a, dn, rng)) {
                    att = vmul(att, a);                                   // main.cu:61
                    o = hp; d = dn;
                    depth++;
                    if (depth >= p.max_depth) sample_done = true;         // main.cu:74
                } else {
                    sample_done = true;                                    // main.cu:64
                }
            } else {
                contrib = vmul(att, sky_h(d));                             // main.cu:68-71
                sample_done = true;
            }
            if (sample_done) {
                col = vadd(col, contrib);                                  // main.cu:107, accumulated in half
                depth = 0;
                s++;
                if (s >= p.ns_local) {
                    float *out = p.out + (size_t)pix * 3;
                    if (p.finalize) {   // main.cu:111-115: col /= real_t(ns); sqrt() is the float one
                        out[0] = h2f(hsqrtf_(hmul_(vx(col), inv_ns)));
                        out[1] = h2f(hsqrtf_(hmul_(vy(col), inv_ns)));
                        out[2] = h2f(hsqrtf_(hmul_(col.z, inv_ns)));
                    } else {
                        out[0] = h2f(vx(col)); out[1] = h2f(vy(col)); out[2] = h2f(col.z);
                    }
                    // main.cu:136: rand_state[pixel_index] = local_rand_state
                    if (PROG && !LIST && p.state_out) xorwow_store(p.state_out + (size_t)pix * 6, rng);
                    if (PROG && LIST) xorwow_store(const_cast<uint32_t *>(p.seed_states) + (size_t)pix * 6, rng);
                    pix = -1;
                }
            }
        }
        __syncwarp();
    }
    unsigned long long r64 = nrays, p64 = npaths;
    for (int off = 16; off > 0; off >>= 1) {
        r64 += __shfl_xor_sync(0xffffffffu, r64, off);
        p64 += __shfl_xor_sync(0xffffffffu, p64, off);
    }
    if (lane == 0) {
        atomicAdd(p.counters + 0, r64);
        atomicAdd(p.counters + 1, p64);
#ifdef RT_COUNTERS
        const CoopSmem &cs = coop_sm[threadIdx.x >> 5];     // two spheres per pair (NaN padding pairs included: they are scanned too)
        atomicAdd(p.counters + 2, 2ull * ((unsigned long long)cs.pairs_hi << 32 | cs.pairs_lo));
#endif
    }
}

// main.cu:111-115 of the USE_FP16 build on linear half sums widened to float (frames assembled from tile shards, progressive
// sums): exactly what k_render_h writes with p.finalize.  Element-wise, so it serves whole frames and reduce-scatter slices.
__global__ void k_finalize_h(const float *__restrict__ accum, float *__restrict__ fb, size_t count, int ns) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) fb[i] = h2f(hsqrtf_(hmul_(f2h(accum[i]), inv_ns_h(ns))));
}

// k_finalize_h with a per-pixel sample count (rt_finalize_counts): what k_render_h writes for a pixel rendered with counts[pix]
// samples; count 0 gives (0, 0, 0)
__global__ void k_finalize_counts_h(const float *__restrict__ accum, const uint32_t *__restrict__ counts, float *__restrict__ fb, size_t npix) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    const uint32_t c = counts[i];
    const float a0 = accum[3 * i], a1 = accum[3 * i + 1], a2 = accum[3 * i + 2];
    if (c == 0) {
        fb[3 * i] = 0.0f; fb[3 * i + 1] = 0.0f; fb[3 * i + 2] = 0.0f;
        return;
    }
    const hf inv_ns = inv_ns_h((int)c);
    fb[3 * i] = h2f(hsqrtf_(hmul_(f2h(a0), inv_ns)));
    fb[3 * i + 1] = h2f(hsqrtf_(hmul_(f2h(a1), inv_ns)));
    fb[3 * i + 2] = h2f(hsqrtf_(hmul_(f2h(a2), inv_ns)));
}

// ---- per-ray queries of the USE_FP16 build: hitTree / hitable_list::hit, camera::get_ray, material::scatter -------------------
// The device functions k_render_h composes, one call per caller-supplied input.  Every float input is rounded to half on entry
// and every output is a half widened to float, so values that came out of one of these kernels go back in exactly.

// Closest hit of n rays: coop_trace_h over the same pair lists, node tables and half slab planes as k_render_h, so the answer is
// the one the render computes.  The warp traces its lanes' rays together (ballots, shuffles, REDUX over the full warp): lanes
// past n stay in the kernel with no ray.  out_t is the hit's half t (+inf on a miss: FLT_MAX rounded to half).  The launch bounds
// are k_render_h's: with kRenderThreads alone ptxas held the octree instance to 56 registers and spilled 46 bytes.
template <bool OCTREE>
__global__ void __launch_bounds__(kRenderThreads, 5)
k_trace_rays_h(const __grid_constant__ RenderLaunch p, const uint2 *__restrict__ geom_h, const PairView pv, const NodeTab nt,
               const float *__restrict__ org, const float *__restrict__ dir, int n, int *__restrict__ out_idx, float *__restrict__ out_t) {
    __shared__ CoopSmem coop_sm[kRenderThreads / 32];
    __shared__ hf planes_h[3 * kPlanes];
    if (OCTREE && threadIdx.x < 3 * kPlanes) planes_h[threadIdx.x] = f2h((&p.tree.planes[0][0])[threadIdx.x]);
    __syncthreads();
    const unsigned lane = threadIdx.x & 31u;
    if (lane == 0) {
        coop_sm[threadIdx.x >> 5].tail = 0u;
        coop_sm[threadIdx.x >> 5].pairs_lo = coop_sm[threadIdx.x >> 5].pairs_hi = 0u;
    }
    __syncwarp();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool have = i < n;
    const hf zero = f2h(0.0f), one = f2h(1.0f);
    vec3h o = mkh(zero, zero, zero), d = mkh(zero, zero, one);
    if (have) {
        o = mkh_f(org[3 * i], org[3 * i + 1], org[3 * i + 2]);
        d = mkh_f(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    }
    const HitH h = coop_trace_h<OCTREE>(coop_sm[threadIdx.x >> 5], planes_h, pv, nt, geom_h, have, o, d);
    if (have) {
        out_idx[i] = h.idx;
        out_t[i] = h2f(h.t);
    }
}

// camera::get_ray (camera.h:45-49) with the context's half camera (22 halves, k_camera_setup_h); each ray draws its lens sample
// from its own XORWOW state (6 words, in and out)
__global__ void k_camera_rays_h(const __half *__restrict__ cam_h, int n, const float *__restrict__ s, const float *__restrict__ t,
                                uint32_t *__restrict__ states, float *__restrict__ org, float *__restrict__ dir) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const CameraH cam = load_camera_h(cam_h);
    uint32_t *st = states + (size_t)i * 6;
    xorwow rng = xorwow_load(st);
    vec3h o, d;
    camera_ray_h(cam, f2h(s[i]), f2h(t[i]), rng, o, d);
    org[3 * i] = h2f(vx(o)); org[3 * i + 1] = h2f(vy(o)); org[3 * i + 2] = h2f(o.z);
    dir[3 * i] = h2f(vx(d)); dir[3 * i + 1] = h2f(vy(d)); dir[3 * i + 2] = h2f(d.z);
    xorwow_store(st, rng);
}

// sphere.h:30-33 + material.h:55-113 for (ray, sphere, t): hit point, normal, scattered direction, attenuation, and
// scattered = 1 / 0 (metal absorbs, material.h:72) / -1 (not a defined sphere); the state is advanced in place
__global__ void k_scatter_rays_h(const uint2 *__restrict__ geom_h, const uint2 *__restrict__ matl_h, const int *__restrict__ tag, int nsph,
                                 int n, const int *__restrict__ sphere_idx, const float *__restrict__ org, const float *__restrict__ dir,
                                 const float *__restrict__ t_hit, uint32_t *__restrict__ states, float *__restrict__ out_p,
                                 float *__restrict__ out_n, float *__restrict__ out_dir, float *__restrict__ out_att, int *__restrict__ scattered) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int idx = sphere_idx[i];
    if (idx < 0 || idx >= nsph || tag[idx] < 0) { scattered[i] = -1; return; }
    uint32_t *st = states + (size_t)i * 6;
    xorwow rng = xorwow_load(st);
    const vec3h o = mkh_f(org[3 * i], org[3 * i + 1], org[3 * i + 2]), d = mkh_f(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    const hf zero = f2h(0.0f);
    vec3h hp, hn, att, dn = mkh(zero, zero, zero);
    hit_point_h(load_sphere_h(geom_h, idx), o, d, f2h(t_hit[i]), hp, hn);
    const bool go = scatter_h(tag[idx], load_mat_h(matl_h, idx), d, hp, hn, att, dn, rng);
    out_p[3 * i] = h2f(vx(hp)); out_p[3 * i + 1] = h2f(vy(hp)); out_p[3 * i + 2] = h2f(hp.z);
    out_n[3 * i] = h2f(vx(hn)); out_n[3 * i + 1] = h2f(vy(hn)); out_n[3 * i + 2] = h2f(hn.z);
    out_dir[3 * i] = h2f(vx(dn)); out_dir[3 * i + 1] = h2f(vy(dn)); out_dir[3 * i + 2] = h2f(dn.z);
    out_att[3 * i] = h2f(vx(att)); out_att[3 * i + 1] = h2f(vy(att)); out_att[3 * i + 2] = h2f(att.z);
    scattered[i] = go ? 1 : 0;
    xorwow_store(st, rng);
}

}  // namespace h16
