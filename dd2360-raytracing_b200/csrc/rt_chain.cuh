// rt_chain.cuh — the lane loop of the persistent FP32 render kernels (k_render, coop::k_render_coop): render + color
// (main.cu:43-117) as one pixel chain per lane.  Included by rt_render.cu inside namespace rt, after the queue and
// seeding helpers it uses (claim_items, item_to_pixel, list_to_pixel, pixel_stream).
//
// Every lane owns one pixel at a time and runs its sample chain bounce by bounce (the chain is inherently serial: all samples
// of a pixel draw from one XORWOW stream, SURVEY D8).  When a lane's pixel is finished it claims the next one (claim_items:
// ballot/popc-compacted, one atomic per warp), so lanes always have a ray to trace, whatever the path lengths of their
// neighbours.  The kernels differ only in how they trace, which they pass to run_chains as a callable; the arithmetic is ChainF32,
// in which every operation is stated explicitly, in the reference's order, so that frames are bit-identical to the reference
// (DESIGN §4).  h16::k_render_h runs the same loop in half precision in a copy of its own: on this body it kept its registers
// but was scheduled differently and rendered C4 1 % slower (B200 at 1000 W).
#pragma once

// The per-lane path state.  pix is the lane's pixel (kModeList: its list slot), -1 while the lane has none.
struct Chain {
    int pix, pi, pj, s, depth;
    xorwow rng;
    vec3f o, d, att, col;
    uint32_t nrays, npaths;
    bool exhausted;
    uint32_t stock_next, stock_end;     // the warp's unclaimed rest of its last tile (claim_items)

    // k_render_coop: what a lane does not need while its warp traces (RNG stream, attenuation, colour sum, pixel bookkeeping:
    // 21 words) is parked in shared memory instead of being spilled to local memory by the register allocator.
    __device__ __forceinline__ void park(uint32_t (*pk)[kRenderThreads], const unsigned t) const {
        pk[0][t] = rng.d; pk[1][t] = rng.v0; pk[2][t] = rng.v1; pk[3][t] = rng.v2; pk[4][t] = rng.v3; pk[5][t] = rng.v4;
        pk[6][t] = __float_as_uint(att.x); pk[7][t] = __float_as_uint(att.y); pk[8][t] = __float_as_uint(att.z);
        pk[9][t] = __float_as_uint(col.x); pk[10][t] = __float_as_uint(col.y); pk[11][t] = __float_as_uint(col.z);
        pk[12][t] = (uint32_t)pi; pk[13][t] = (uint32_t)pj; pk[14][t] = (uint32_t)s; pk[15][t] = (uint32_t)depth;
        pk[16][t] = (uint32_t)pix; pk[17][t] = nrays; pk[18][t] = npaths; pk[19][t] = stock_next; pk[20][t] = stock_end;
    }
    __device__ __forceinline__ void unpark(uint32_t (*pk)[kRenderThreads], const unsigned t) {
        rng.d = pk[0][t]; rng.v0 = pk[1][t]; rng.v1 = pk[2][t]; rng.v2 = pk[3][t]; rng.v3 = pk[4][t]; rng.v4 = pk[5][t];
        att = mk(__uint_as_float(pk[6][t]), __uint_as_float(pk[7][t]), __uint_as_float(pk[8][t]));
        col = mk(__uint_as_float(pk[9][t]), __uint_as_float(pk[10][t]), __uint_as_float(pk[11][t]));
        pi = (int)pk[12][t]; pj = (int)pk[13][t]; s = (int)pk[14][t]; depth = (int)pk[15][t];
        pix = (int)pk[16][t]; nrays = pk[17][t]; npaths = pk[18][t]; stock_next = pk[19][t]; stock_end = pk[20][t];
    }
};

// The reference's float build (vec3.h, camera.h, material.h).
struct ChainF32 {
    typedef vec3f V;
    const RenderLaunch &p;
    float inv_ns;
    __device__ __forceinline__ explicit ChainF32(const RenderLaunch &p_) : p(p_) { inv_ns = __fdiv_rn(1.0f, (float)p.ns_total); }   // vec3.h:137-144: k = 1.0/t

    __device__ __forceinline__ V vec(float x, float y, float z) const { return mk(x, y, z); }
    __device__ __forceinline__ V mul(const V a, const V b) const { return mk(mul_(a.x, b.x), mul_(a.y, b.y), mul_(a.z, b.z)); }
    __device__ __forceinline__ V add(const V a, const V b) const { return mk(add_(a.x, b.x), add_(a.y, b.y), add_(a.z, b.z)); }
    __device__ __forceinline__ V sky(const V d) const { return ::rt::sky(d); }
    // main.cu:104-106
    __device__ __forceinline__ void camera(const int pi, const int pj, xorwow &rng, V &o, V &d) const {
        const float u = div_(add_((float)pi, xorwow_uniform(rng)), (float)p.nx);
        const float v = div_(add_((float)pj, xorwow_uniform(rng)), (float)p.ny);
        camera_ray(p.cam, u, v, rng, o, d);
    }
    __device__ __forceinline__ bool scatter(const Hit &h, const V o, const V d, V &hp, V &hn, V &a, V &dn, xorwow &rng) const {
        const float4 g = __ldg(p.scene.geom + h.idx);
        const float4 m = __ldg(p.scene.matl + h.idx);
        const int tag = __ldg(p.scene.tag + h.idx);
        hit_point(g, o, d, h.t, hp, hn);
        return ::rt::scatter(tag, m, d, hp, hn, a, dn, rng);
    }
    __device__ __forceinline__ void write(float *out, const V col) const {
        if (p.finalize) {   // main.cu:111-115
            out[0] = sqrt_(mul_(col.x, inv_ns));
            out[1] = sqrt_(mul_(col.y, inv_ns));
            out[2] = sqrt_(mul_(col.z, inv_ns));
        } else {
            out[0] = col.x; out[1] = col.y; out[2] = col.z;
        }
    }
};

// Runs the lanes of one warp until the queue is exhausted, then adds their ray and path counts to p.counters[0..1].
// trace(chain, has) returns the closest hit of the chain's ray (o, d); every lane of the warp calls it, `has` says whether the
// lane holds a pixel, and it may reload the chain (k_render_coop parks it).  batch: claim_items' tile batch.
// MODE (rt_render.h LaunchMode) says what the queue's items are:
//   kModeFrame: 8x4 tiles of the frame; progressive calls continue the sum in `out` (p.accumulate) and store the stream to
//               p.state_out;
//   kModeList: list entries, each rendered from sample 0 into its list slot (the list pointer shares state_out's slot);
//   kModeListProgressive: list entries, each a FRAME pixel: its sum continues in out[3 * pixel] (p.accumulate) and its stream is
//               resumed from and stored back to seed_states[6 * pixel].  The list is deduplicated (k_pixels_progressive_prep),
//               so no two lanes hold one pixel; an entry outside the frame is skipped and writes nothing.
template <int MODE, class Trace>
__device__ __forceinline__ void run_chains(const RenderLaunch &p, const ChainF32 &pol, const uint32_t batch, Trace &&trace) {
    const unsigned lane = threadIdx.x & 31u;
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    Chain c;
    c.pix = -1; c.pi = 0; c.pj = 0; c.s = 0; c.depth = 0;
    c.rng.d = c.rng.v0 = c.rng.v1 = c.rng.v2 = c.rng.v3 = c.rng.v4 = 0;
    c.o = pol.vec(0.f, 0.f, 0.f); c.d = pol.vec(0.f, 0.f, 1.f); c.att = pol.vec(1.f, 1.f, 1.f); c.col = pol.vec(0.f, 0.f, 0.f);
    c.nrays = 0; c.npaths = 0;
    c.exhausted = false;
    c.stock_next = gwarp * 32u; c.stock_end = c.stock_next + 32u;   // the first tile needs no atomic: the queue head starts past the grid

    while (true) {
        // ---- claim pixels for idle lanes ----
        while (true) {
            const bool need = c.pix < 0 && !c.exhausted;
            const unsigned m = __ballot_sync(0xffffffffu, need);
            if (!m) break;
            const uint32_t item = claim_items(p, m, lane, c.stock_next, c.stock_end, batch);
            if (need) {
                if (item >= p.total_items) {
                    c.exhausted = true;
                } else if (MODE != kModeFrame ? list_to_pixel(p, item, c.pi, c.pj, MODE == kModeList) : item_to_pixel(p, item, c.pi, c.pj)) {
                    c.pix = MODE == kModeList ? (int)item : c.pj * p.nx + c.pi;
                    c.s = 0; c.depth = 0;
                    c.col = pol.vec(0.f, 0.f, 0.f);
                    if (MODE != kModeList && p.accumulate) {   // progressive: continue the pixel's sum exactly where the last call left it
                        const float *acc = p.out + (size_t)c.pix * 3;
                        c.col = pol.vec(acc[0], acc[1], acc[2]);
                    }
                    pixel_stream(p, MODE == kModeList && !p.seed_states ? c.pj * p.nx + c.pi : c.pix, c.rng);
                }
            }
        }
        if (!__ballot_sync(0xffffffffu, c.pix >= 0)) break;

        const bool has = c.pix >= 0;
        if (has) {
            if (c.depth == 0) {   // new sample: main.cu:104-106
                pol.camera(c.pi, c.pj, c.rng, c.o, c.d);
                c.att = pol.vec(1.f, 1.f, 1.f);
                c.npaths++;
            }
            c.nrays++;
        }
        const auto h = trace(c, has);
        // (c.pix, not `has`: a parking trace reloads pix, and keeping `has` live across coop_trace costs k_render_coop stack)
        if (c.pix >= 0) {   // ---- one iteration of color()'s loop (main.cu:47-73) ----
            bool sample_done = false;
            vec3f contrib = pol.vec(0.f, 0.f, 0.f);
            if (h.idx >= 0) {
                vec3f hp, hn, a, dn;
                if (pol.scatter(h, c.o, c.d, hp, hn, a, dn, c.rng)) {
                    c.att = pol.mul(c.att, a);                               // main.cu:61
                    c.o = hp; c.d = dn;
                    c.depth++;
                    if (c.depth >= p.max_depth) sample_done = true;          // main.cu:74: return black
                } else {
                    sample_done = true;                                      // absorbed: main.cu:64
                }
            } else {
                contrib = pol.mul(c.att, pol.sky(c.d));                      // main.cu:68-71
                sample_done = true;
            }
            if (sample_done) {
                c.col = pol.add(c.col, contrib);                             // main.cu:107
                c.depth = 0;
                c.s++;
                if (c.s >= p.ns_local) {
                    pol.write(p.out + (size_t)c.pix * 3, c.col);
                    // main.cu:136: rand_state[pixel_index] = local_rand_state
                    if (MODE == kModeFrame && p.state_out) xorwow_store(p.state_out + (size_t)c.pix * 6, c.rng);
                    if (MODE == kModeListProgressive) xorwow_store(const_cast<uint32_t *>(p.seed_states) + (size_t)c.pix * 6, c.rng);
                    c.pix = -1;
                }
            }
        }
        __syncwarp();
    }

    // ---- ray / path counters: one atomic per warp ----
    unsigned long long r64 = c.nrays, p64 = c.npaths;
    for (int off = 16; off > 0; off >>= 1) {
        r64 += __shfl_xor_sync(0xffffffffu, r64, off);
        p64 += __shfl_xor_sync(0xffffffffu, p64, off);
    }
    if (lane == 0) {
        atomicAdd(p.counters + 0, r64);
        atomicAdd(p.counters + 1, p64);
    }
}
