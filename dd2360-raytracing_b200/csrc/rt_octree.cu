// rt_octree.cu — parallel GPU build of (a) the traversal structure the render kernel uses and (b) the tree in the
// reference's own memory layout, bit-exact against the serial buildOctree (acceleration_structure.h:195-217).
//
// Pipeline (one stream; three small read-backs size the allocations):
//   k_classify      sphere -> per-axis level-3 slab ranges (reference `intersects` semantics), entry count,
//                   per-cell histogram (shared-memory privatised)
//   scan            entry offsets (also the per-sphere cell lists of VisView)       (cub::DeviceScan)
//   k_emit          (Morton cell key, sphere index) pairs in sphere order
//   radix sort      stable, 9 key bits -> cell-major, sphere-ascending              (cub::DeviceRadixSort)
//   k_mark_entries  in-cell rank -> which entries the reference drops ("Leaf nodes full"), which spheres are stored
//   k_number_nodes  one block: first-touch numbering of the nodes = the serial creation order
//   k_grid_prep     big/small split, bounding box and count of the spheres that go into the grid
//   (host)          grid resolution
//   k_vox_pass x2 + scan + k_vox_finish   sphere-surface x voxel incidence lists, sorted, {start,count} per voxel
//   (on export)     k_leaf_number, k_blob_nodes, k_blob_leaves -> reference `Octree` blob
// CUB (shipped inside the CUDA toolkit, header-only) provides the device-wide scan and radix sort; everything
// else is hand-written.
#include <cub/cub.cuh>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <limits.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "rt_build.cuh"
#include "rt_octree.h"

namespace rt {

#define RT_CUDA(x)                          \
    do {                                    \
        cudaError_t e_ = (x);               \
        if (e_ != cudaSuccess) return e_;   \
    } while (0)

// acceleration_structure.h:82-93 along one axis under USE_FP16: centre, radius and box are halves, the grown bounds round to half
__device__ __forceinline__ AxisRange axis_range_h(const float *P, float c, float r, bool open_low) {
    AxisRange a;
    a.lo = 8; a.hi = -1;
    const __half ch = __float2half_rn(c), rh = __float2half_rn(r);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const __half low = __hsub_rn(__float2half_rn(P[i]), rh), high = __hadd_rn(__float2half_rn(P[i + 1]), rh);
        const bool in = (open_low ? __hgt(ch, low) : __hge(ch, low)) && __hle(ch, high);
        if (in) { a.lo = imin(a.lo, i); a.hi = imax(a.hi, i); }
    }
    return a;
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void k_classify(const float4 *__restrict__ geom, int n, BuildPlanes P, int fp16, uint32_t *__restrict__ ranges,
                           uint32_t *__restrict__ ent_count, uint32_t *__restrict__ cell_count,
                           unsigned long long *__restrict__ dropped_outside) {
    __shared__ uint32_t hist[kCells];
    for (int k = threadIdx.x; k < kCells; k += blockDim.x) hist[k] = 0;
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        uint32_t packed = 0, cnt = 0;
        if (i >= 1) {   // ground sphere (index 0) is never inserted (acceleration_structure.h:208)
            const float4 s = geom[i];
            // the SIGNED radius, as `intersects` has it: a cell shrinks by |r| for a hollow sphere (r < 0), so one with |r| >= 0.125
            // (half a cell's height) is stored nowhere and smaller ones only where the centre lies.  The grid lists surfaces: |r|.
            // USE_FP16: AABB, centre and radius are real_t, so `low - radius` / `high + radius` round to half
            // (acceleration_structure.h:83-88); the planes themselves are exact in half
            const AxisRange rx = fp16 ? axis_range_h(P.p[0], s.x, s.w, true) : axis_range(P.p[0], s.x, s.w, true);
            const AxisRange ry = fp16 ? axis_range_h(P.p[1], s.y, s.w, false) : axis_range(P.p[1], s.y, s.w, false);
            const AxisRange rz = fp16 ? axis_range_h(P.p[2], s.z, s.w, false) : axis_range(P.p[2], s.z, s.w, false);
            if (rx.lo <= rx.hi && ry.lo <= ry.hi && rz.lo <= rz.hi) {
                cnt = (uint32_t)((rx.hi - rx.lo + 1) * (ry.hi - ry.lo + 1) * (rz.hi - rz.lo + 1));
                packed = 1u << 31 | rx.lo | rx.hi << 4 | ry.lo << 8 | ry.hi << 12 | rz.lo << 16 | rz.hi << 20;
                for (int x = rx.lo; x <= rx.hi; x++)
                    for (int y = ry.lo; y <= ry.hi; y++)
                        for (int z = rz.lo; z <= rz.hi; z++) atomicAdd(&hist[morton_of(x, y, z)], 1u);
            } else {
                atomicAdd(dropped_outside, 1ull);   // ":105-108 Why is sphere not in range of nodes AABB?"
            }
        }
        ranges[i] = packed;
        ent_count[i] = cnt;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kCells; k += blockDim.x)
        if (hist[k]) atomicAdd(&cell_count[k], hist[k]);
}

__global__ void k_emit(const uint32_t *__restrict__ ranges, const uint32_t *__restrict__ ent_off, int n,
                       uint32_t *__restrict__ keys, uint32_t *__restrict__ vals, uint16_t *__restrict__ ent_cell) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t p = ranges[i];
    if (!(p >> 31)) return;
    uint32_t o = ent_off[i];
    const int xl = p & 15, xh = (p >> 4) & 15, yl = (p >> 8) & 15, yh = (p >> 12) & 15, zl = (p >> 16) & 15, zh = (p >> 20) & 15;
    for (int x = xl; x <= xh; x++)
        for (int y = yl; y <= yh; y++)
            for (int z = zl; z <= zh; z++) {
                const uint32_t m = (uint32_t)morton_of(x, y, z);
                keys[o] = m;
                vals[o] = (uint32_t)i;
                ent_cell[o] = (uint16_t)m;      // sphere-major: the cells sphere i was inserted into (VisView)
                o++;
            }
}

// exclusive scan of the 512 cell counts (one block of 512 threads)
__global__ void k_cell_scan(const uint32_t *__restrict__ cell_count, uint32_t *__restrict__ cell_start) {
    __shared__ uint32_t s[kCells];
    const int t = threadIdx.x;
    s[t] = cell_count[t];
    __syncthreads();
    for (int off = 1; off < kCells; off <<= 1) {
        uint32_t v = t >= off ? s[t - off] : 0;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    cell_start[t + 1] = s[t];
    if (t == 0) cell_start[0] = 0;
}

// Per sorted entry: the reference stores the first 8*SPL entries of a cell and drops the rest (:110-136).
__global__ void k_mark_entries(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                               const uint32_t *__restrict__ cell_start, uint32_t E, int spl,
                               const uint32_t *__restrict__ ranges, const uint32_t *__restrict__ ent_off,
                               uint16_t *__restrict__ ent_cell, uint8_t *__restrict__ sph_flag,
                               unsigned long long *__restrict__ stats /* [0] stored, [1] dropped_full */) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    bool stored = false, dropped = false;
    if (p < E) {
        const uint32_t m = keys[p], S = vals[p];
        const uint32_t pos = p - cell_start[m];
        dropped = pos >= 8u * (uint32_t)spl;
        stored = !dropped;
        if (dropped) {
            // locate this entry in the sphere's own (x, y, z)-ordered list
            const uint32_t r = ranges[S];
            const int yl = (r >> 8) & 15, yh = (r >> 12) & 15, zl = (r >> 16) & 15, zh = (r >> 20) & 15, xl = r & 15;
            int ix, iy, iz;
            morton_to_xyz((int)m, ix, iy, iz);
            const uint32_t local = (uint32_t)(((ix - xl) * (yh - yl + 1) + (iy - yl)) * (zh - zl + 1) + (iz - zl));
            ent_cell[ent_off[S] + local] = (uint16_t)(m | kEntDropped);
        } else {
            sph_flag[S] = 1;          // stored in at least one cell (benign race: every writer writes 1)
        }
    }
    const unsigned ms = __ballot_sync(0xffffffffu, stored), md = __ballot_sync(0xffffffffu, dropped);
    if ((threadIdx.x & 31) == 0) {
        if (ms) atomicAdd(&stats[0], (unsigned long long)__popc(ms));
        if (md) atomicAdd(&stats[1], (unsigned long long)__popc(md));
    }
}

// One block (1024 threads): number the nodes in the reference's creation order.
__global__ void k_number_nodes(const uint32_t *__restrict__ vals, const uint32_t *__restrict__ cell_start,
                               int *__restrict__ node_of_potential, BuildCounts *__restrict__ out) {
    __shared__ int first[kNumberNodes];      // first sphere index touching the potential node
    const int t = threadIdx.x;
    if (t < kCells) {
        const uint32_t b = cell_start[t], e = cell_start[t + 1];
        first[level_base(3) + t] = e > b ? (int)vals[b] : INT_MAX;   // lists ascend, so the head is the first toucher
    }
    __syncthreads();
    if (t < 64) { int f = INT_MAX; for (int c = 0; c < 8; c++) f = min(f, first[level_base(3) + t * 8 + c]); first[level_base(2) + t] = f; }
    __syncthreads();
    if (t < 8) { int f = INT_MAX; for (int c = 0; c < 8; c++) f = min(f, first[level_base(2) + t * 8 + c]); first[level_base(1) + t] = f; }
    __syncthreads();
    if (t == 0) first[0] = -1;   // the root always exists and is created before any insertion (:200-206)
    __syncthreads();
    // creation order = sort by (first toucher, pre-order position); rank by counting (585^2 compares)
    if (t < kNumberNodes) {
        const int my_level = t >= level_base(3) ? 3 : (t >= level_base(2) ? 2 : (t >= level_base(1) ? 1 : 0));
        int rank = -1;
        if (first[t] != INT_MAX) {
            const long long mykey = (long long)first[t] * 4096 + preorder_key(my_level, t - level_base(my_level));
            rank = 0;
            for (int j = 0; j < kNumberNodes; j++) {
                if (first[j] == INT_MAX) continue;
                const int lv = j >= level_base(3) ? 3 : (j >= level_base(2) ? 2 : (j >= level_base(1) ? 1 : 0));
                rank += ((long long)first[j] * 4096 + preorder_key(lv, j - level_base(lv))) < mykey;
            }
        }
        node_of_potential[t] = rank;
    }
    if (t == 0) {
        int nc = 0;
        for (int j = 0; j < kNumberNodes; j++) nc += first[j] != INT_MAX;
        out->node_count = nc;
    }
}

// order-preserving float <-> uint map, so that atomicMin/atomicMax on uints order floats
__device__ __forceinline__ uint32_t f2ord(float f) { const uint32_t b = __float_as_uint(f); return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u); }
inline float ord2f(uint32_t o) { const uint32_t b = o ^ ((o >> 31) ? 0x80000000u : 0xffffffffu); float f; memcpy(&f, &b, 4); return f; }

// Which spheres go into the grid, which are "big", and the bounding box of the gridded ones.
// sph_flag: 0 = not traceable (undefined slot, outside the root box, or every entry dropped), 1 = gridded, 2 = big.
__global__ void k_grid_prep(const float4 *__restrict__ geom, const int *__restrict__ tag, int n, float big_r,
                            uint8_t *__restrict__ sph_flag, GridPrep *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f};
    uint32_t live = 0;
    if (i < n) {
        if (i == 0) out->slot0_none = tag[0] < 0 ? 1u : 0u;
        uint8_t f = sph_flag[i];
        if (f && tag[i] < 0) f = 0;                       // undefined slots are never hit (SURVEY D3)
        if (f) {
            const float4 s = geom[i];
            const float ar = fabsf(s.w);                  // a hollow sphere (r < 0) is hit where |r| puts its surface (r*r)
            if (ar > big_r) {
                const uint32_t slot = atomicAdd(&out->nbig, 1u);
                if (slot < (uint32_t)kMaxBig) { out->big[slot] = (uint32_t)i; f = 2; }
            }
            if (f == 1) {
                const float r = ar + sphere_pad(ar);
                lo[0] = s.x - r; hi[0] = s.x + r; lo[1] = s.y - r; hi[1] = s.y + r; lo[2] = s.z - r; hi[2] = s.z + r;
                live = 1;
            }
        }
        sph_flag[i] = f;
    }
    for (int o = 16; o > 0; o >>= 1) {
        for (int k = 0; k < 3; k++) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(0xffffffffu, lo[k], o));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(0xffffffffu, hi[k], o));
        }
        live += __shfl_xor_sync(0xffffffffu, live, o);
    }
    if ((threadIdx.x & 31) == 0 && live) {
        for (int k = 0; k < 3; k++) { atomicMin(&out->lo[k], f2ord(lo[k])); atomicMax(&out->hi[k], f2ord(hi[k])); }
        atomicAdd(&out->live, live);
    }
}

// enumerate the voxels crossed by the (padded) surface of sphere s; a hollow sphere (r < 0) by |r|
template <typename F>
__device__ __forceinline__ void for_each_voxel(const GridView &g, float4 s, F f) {
    s.w = fabsf(s.w);
    const float pad = sphere_pad(s.w);
    int v0[3], v1[3];
    voxel_range(g, s, pad, v0, v1);
    for (int z = v0[2]; z <= v1[2]; z++)
        for (int y = v0[1]; y <= v1[1]; y++)
            for (int x = v0[0]; x <= v1[0]; x++) {
                float lo[3], hi[3];
                voxel_box(g, x, y, z, lo, hi);
                if (shell_hits_box(s, pad, lo, hi)) f((uint32_t)(((size_t)z * g.ny + y) * g.nx + x));
            }
}

template <bool FILL>
__global__ void k_vox_pass(const float4 *__restrict__ geom, const uint8_t *__restrict__ sph_flag, int n,
                           const __grid_constant__ GridView g, uint32_t *__restrict__ counter,
                           const uint32_t *__restrict__ vox_start, uint32_t *__restrict__ refs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || sph_flag[i] != 1) return;
    const float4 s = geom[i];
    for_each_voxel(g, s, [&](uint32_t v) {
        const uint32_t slot = atomicAdd(&counter[v], 1u);
        if (FILL) refs[vox_start[v] + slot] = (uint32_t)i;
    });
}

// per voxel: ascending order (deterministic traversal) and the {start, count} record the render kernel reads
__global__ void k_vox_finish(const uint32_t *__restrict__ vox_start, uint32_t total_voxels, uint32_t *__restrict__ refs,
                             uint2 *__restrict__ vox) {
    const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= total_voxels) return;
    const uint32_t b = vox_start[v], e = vox_start[v + 1];
    for (uint32_t a = b + 1; a < e; a++) {
        const uint32_t x = refs[a];
        uint32_t j = a;
        while (j > b && refs[j - 1] > x) { refs[j] = refs[j - 1]; j--; }
        refs[j] = x;
    }
    vox[v] = make_uint2(b, e - b);
}

// geometry in list order (TreeView::ref_geom / prolog_geom)
__global__ void k_gather_geom(const float4 *__restrict__ geom, const uint32_t *__restrict__ refs, size_t count, float4 *__restrict__ out) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < count) out[k] = geom[refs[k]];
}

// ---- reference-layout blob ------------------------------------------------------------------------------------
// bucket (cell m, slot k) exists when k*spl < stored(m); its creator is the sphere with in-cell rank k*spl.
__global__ void k_leaf_number(const uint32_t *__restrict__ vals, const uint32_t *__restrict__ cell_start, int spl,
                              int *__restrict__ leaf_index /* [512*8] */, int *__restrict__ leaf_count) {
    const int id = blockIdx.x * blockDim.x + threadIdx.x;   // m*8 + k
    if (id >= kCells * 8) return;
    auto key_of = [&](int j) -> long long {
        const int m = j >> 3, k = j & 7;
        const uint32_t b = cell_start[m], e = cell_start[m + 1];
        const uint32_t count = e - b, cap = 8u * (uint32_t)spl;
        const uint32_t stored = count < cap ? count : cap;
        if ((uint32_t)k * (uint32_t)spl >= stored) return -1;
        return ((long long)vals[b + (uint32_t)k * (uint32_t)spl] << 12) | preorder_key(3, m);
    };
    const long long mykey = key_of(id);
    int rank = -1;
    if (mykey >= 0) {
        rank = 0;
        for (int j = 0; j < kCells * 8; j++) {
            const long long kj = key_of(j);
            rank += (kj >= 0 && kj < mykey);
        }
        atomicAdd(leaf_count, 1);
    }
    leaf_index[id] = rank >= 0 ? rank + 1 : 0;   // leaves[0] is never used (:58)
}

// OctNode (acceleration_structure.h:34-38) = {int level, AABB, int children[8]}.  AABB is six real_t: floats (60-byte nodes), or
// under USE_FP16 halves (48-byte nodes: level at 0, the box at 4, children at 16).  The box planes are multiples of 2.75 (x, z)
// and 0.25 (y) in [-11, 11], exact in half, and so is the reference's half subdivision low + (high - low) / 2 of exact values:
// the half AABB is the float plane rounded to half.  rt_octree_export_reference checks that every plane round-trips.
template <bool HALF>
__global__ void k_blob_nodes(const int *__restrict__ node_of_potential, const int *__restrict__ leaf_index,
                             BuildPlanes P, uint8_t *__restrict__ blob_nodes) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= kNumberNodes) return;
    const int ni = node_of_potential[t];
    if (ni < 0) return;
    const int lv = t >= level_base(3) ? 3 : (t >= level_base(2) ? 2 : (t >= level_base(1) ? 1 : 0));
    const int path = t - level_base(lv);
    int ix = 0, iy = 0, iz = 0;
    for (int l = 0; l < lv; l++) {
        const int c = (path >> (3 * (lv - 1 - l))) & 7;
        ix = (ix << 1) | (c >> 2); iy = (iy << 1) | ((c >> 1) & 1); iz = (iz << 1) | (c & 1);
    }
    const int sh = 3 - lv;
    uint8_t *nd = blob_nodes + (size_t)ni * (HALF ? kNodeBytesHalf : kNodeInts * 4);
    *reinterpret_cast<int32_t *>(nd) = lv;
    const float box[6] = {P.p[0][ix << sh], P.p[1][iy << sh], P.p[2][iz << sh],
                          P.p[0][(ix + 1) << sh], P.p[1][(iy + 1) << sh], P.p[2][(iz + 1) << sh]};
    if (HALF) {
        __half *bx = reinterpret_cast<__half *>(nd + 4);
        for (int k = 0; k < 6; k++) bx[k] = __float2half_rn(box[k]);
    } else {
        float *bx = reinterpret_cast<float *>(nd + 4);
        for (int k = 0; k < 6; k++) bx[k] = box[k];
    }
    int32_t *children = reinterpret_cast<int32_t *>(nd + 4 + 6 * (HALF ? 2 : 4));
    for (int c = 0; c < 8; c++) {
        int v;
        if (lv < 3) { const int ch = node_of_potential[level_base(lv + 1) + path * 8 + c]; v = ch >= 0 ? ch : 0; }
        else v = leaf_index[path * 8 + c];
        children[c] = v;
    }
}

__global__ void k_blob_leaves(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                              const uint32_t *__restrict__ cell_start, uint32_t E, int spl,
                              const int *__restrict__ leaf_index, int32_t *__restrict__ blob_leaves) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= E) return;
    const uint32_t m = keys[p];
    const uint32_t b = cell_start[m], e = cell_start[m + 1];
    const uint32_t pos = p - b, count = e - b, cap = 8u * (uint32_t)spl;
    if (pos >= cap) return;                                   // "Leaf nodes full" (:135)
    const uint32_t stored = count < cap ? count : cap;
    const uint32_t k = pos / (uint32_t)spl, slot = pos % (uint32_t)spl;
    int32_t *lf = blob_leaves + (size_t)leaf_index[m * 8 + k] * (size_t)(spl + 1);
    lf[slot] = (int32_t)vals[p];
    if (slot == 0) {
        const uint32_t left = stored - k * (uint32_t)spl;
        lf[spl] = (int32_t)(left < (uint32_t)spl ? left : (uint32_t)spl);
    }
}

// ---------------------------------------------------------------------------------------------------------------
static void make_planes(BuildPlanes &P) {
    // acceleration_structure.h:141-147,203: root (-11,0,-11)-(11,2,11), children by low + (high-low)/2 in float
    const float lo[3] = {-11.f, 0.f, -11.f}, hi[3] = {11.f, 2.f, 11.f};
    for (int a = 0; a < 3; a++) {
        float *p = P.p[a];
        p[0] = lo[a]; p[8] = hi[a];
        for (int step = 8; step > 1; step >>= 1)
            for (int i = 0; i < 8; i += step) {
                volatile float l = p[i], h = p[i + step];
                volatile float d = h - l;
                volatile float half = d / 2;
                p[i + step / 2] = l + half;
            }
    }
}

// the arrays sized by the scene grow with headroom, so that rebuilds of slightly larger scenes reuse them
template <typename T>
static cudaError_t ensure(Buffer<T> &b, size_t need) {
    return b.reserve(need, need / 4 + 256);
}

OctreeBuilder::OctreeBuilder() : grid_flat(kGridFlat), grid_wide(kGridWide), grid_flat_min(kFlatVoxelMinSpheres) {
    memset(&grid, 0, sizeof grid); make_planes(planes);
}

// RT_BUILD_TRACE=1: host wall clock at the build's synchronisation points (diagnostic, stderr)
struct BuildTrace {
    bool on;
    std::chrono::steady_clock::time_point t0;
    BuildTrace() : on(getenv("RT_BUILD_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char *what) {
        if (!on) return;
        const double us = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count();
        fprintf(stderr, "[build] %-28s %9.1f us\n", what, us);
    }
};

cudaError_t OctreeBuilder::build(cudaStream_t st, const float4 *geom, const int *tag, int n, int spl_, float density, bool fp16_,
                                 bool all_spheres_) {
    BuildTrace trace;
    spl = spl_;
    fp16 = fp16_;
    all_spheres = all_spheres_;
    built = false;
    blob_valid = false;
    RT_CUDA(ensure(d.ranges, (size_t)n + 1));
    RT_CUDA(ensure(d.ent_count, (size_t)n + 1));
    RT_CUDA(ensure(d.ent_off, (size_t)n + 1));
    RT_CUDA(ensure(d.sph_flag, (size_t)n + 1));
    RT_CUDA(d.cell_count.reserve(kCells));
    RT_CUDA(d.cell_start.reserve(kCells + 1));
    RT_CUDA(d.stats.reserve(4));
    RT_CUDA(d.node_of_potential.reserve(kNumberNodes));
    RT_CUDA(d.counts.reserve(1));
    RT_CUDA(d.prep.reserve(1));
    RT_CUDA(d.big_refs.reserve(kMaxBig + 1));   // [0] = ground sphere, then the big spheres
    RT_CUDA(d.leaf_index.reserve(kCells * 8 + 1));
    RT_CUDA(cudaMemsetAsync(d.cell_count.ptr, 0, kCells * 4, st));
    RT_CUDA(cudaMemsetAsync(d.stats.ptr, 0, 4 * 8, st));
    RT_CUDA(cudaMemsetAsync(d.ent_count.ptr + n, 0, 4, st));
    RT_CUDA(cudaMemsetAsync(d.sph_flag.ptr, 0, (size_t)n + 1, st));
    const int tb = 256;
    k_classify<<<(n + tb - 1) / tb, tb, 0, st>>>(geom, n, planes, fp16 ? 1 : 0, d.ranges.ptr, d.ent_count.ptr, d.cell_count.ptr, d.stats.ptr + 2);
    size_t tmp = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp, d.ent_count.ptr, d.ent_off.ptr, n + 1, st);
    RT_CUDA(ensure(d.cub_tmp, tmp));
    cub::DeviceScan::ExclusiveSum(d.cub_tmp.ptr, tmp, d.ent_count.ptr, d.ent_off.ptr, n + 1, st);
    uint32_t E_h = 0;
    RT_CUDA(cudaMemcpyAsync(&E_h, d.ent_off.ptr + n, 4, cudaMemcpyDeviceToHost, st));
    trace.mark("classify+scan issued");
    RT_CUDA(cudaStreamSynchronize(st));
    trace.mark("sync 1 (entry count)");
    E = E_h;
    RT_CUDA(ensure(d.keys, (size_t)E + 1));
    RT_CUDA(ensure(d.vals, (size_t)E + 1));
    RT_CUDA(ensure(d.keys_sorted, (size_t)E + 1));
    RT_CUDA(ensure(d.vals_sorted, (size_t)E + 1));
    RT_CUDA(ensure(d.ent_cell, (size_t)E + 2));
    k_emit<<<(n + tb - 1) / tb, tb, 0, st>>>(d.ranges.ptr, d.ent_off.ptr, n, d.keys.ptr, d.vals.ptr, d.ent_cell.ptr);
    if (E > 0) {
        tmp = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp, d.keys.ptr, d.keys_sorted.ptr, d.vals.ptr, d.vals_sorted.ptr, (int)E, 0, 9, st);
        RT_CUDA(ensure(d.cub_tmp, tmp));
        cub::DeviceRadixSort::SortPairs(d.cub_tmp.ptr, tmp, d.keys.ptr, d.keys_sorted.ptr, d.vals.ptr, d.vals_sorted.ptr, (int)E, 0, 9, st);
    }
    k_cell_scan<<<1, kCells, 0, st>>>(d.cell_count.ptr, d.cell_start.ptr);
    if (E > 0)
        k_mark_entries<<<(E + tb - 1) / tb, tb, 0, st>>>(d.keys_sorted.ptr, d.vals_sorted.ptr, d.cell_start.ptr, E, spl, d.ranges.ptr,
                                                        d.ent_off.ptr, d.ent_cell.ptr, d.sph_flag.ptr, d.stats.ptr);
    k_number_nodes<<<1, 1024, 0, st>>>(d.vals_sorted.ptr, d.cell_start.ptr, d.node_of_potential.ptr, d.counts.ptr);
    // grid over the small stored spheres
    GridPrep init;
    memset(&init, 0, sizeof init);
    for (int k = 0; k < 3; k++) { init.lo[k] = 0xffffffffu; init.hi[k] = 0u; }
    RT_CUDA(cudaMemcpyAsync(d.prep.ptr, &init, sizeof init, cudaMemcpyHostToDevice, st));
    const float big_r = kBigRadiusFrac * fmaxf(planes.p[0][1] - planes.p[0][0], fmaxf(planes.p[1][1] - planes.p[1][0], planes.p[2][1] - planes.p[2][0]));
    if (all_spheres) RT_CUDA(cudaMemsetAsync(d.sph_flag.ptr + 1, 1, (size_t)n - 1, st));     // every sphere but the ground (prolog[0])
    k_grid_prep<<<(n + tb - 1) / tb, tb, 0, st>>>(geom, tag, n, big_r, d.sph_flag.ptr, d.prep.ptr);
    GridPrep prep;
    RT_CUDA(cudaMemcpyAsync(&prep, d.prep.ptr, sizeof prep, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaMemcpyAsync(&counts, d.counts.ptr, sizeof counts, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaMemcpyAsync(stats_h, d.stats.ptr, 4 * 8, cudaMemcpyDeviceToHost, st));
    trace.mark("sort..grid_prep issued");
    RT_CUDA(cudaStreamSynchronize(st));
    trace.mark("sync 2 (counts, grid box)");
    nbig = (int)(prep.nbig < (uint32_t)kMaxBig ? prep.nbig : (uint32_t)kMaxBig);
    slot0_none = prep.slot0_none != 0u ? 1 : 0;
    std::sort(prep.big, prep.big + nbig);       // ascending: deterministic traversal order
    prolog_h[0] = 0;
    memcpy(prolog_h + 1, prep.big, kMaxBig * 4);
    RT_CUDA(cudaMemcpyAsync(d.big_refs.ptr, prolog_h, (kMaxBig + 1) * 4, cudaMemcpyHostToDevice, st));
    float lo[3], hi[3];
    for (int k = 0; k < 3; k++) { lo[k] = ord2f(prep.lo[k]); hi[k] = ord2f(prep.hi[k]); }
    memset(&grid, 0, sizeof grid);
    const uint32_t V = choose_grid(lo, hi, prep.live, density, grid, grid_flat, grid_wide, grid_flat_min);
    total_voxels = V;
    total_refs = 0;
    RT_CUDA(ensure(d.vox_count, (size_t)V + 2));
    RT_CUDA(ensure(d.vox_start, (size_t)V + 2));
    RT_CUDA(ensure(d.vox, (size_t)V + 1));
    if (V > 0) {
        RT_CUDA(cudaMemsetAsync(d.vox_count.ptr, 0, ((size_t)V + 2) * 4, st));
        k_vox_pass<false><<<(n + tb - 1) / tb, tb, 0, st>>>(geom, d.sph_flag.ptr, n, grid, d.vox_count.ptr, nullptr, nullptr);
        tmp = 0;
        cub::DeviceScan::ExclusiveSum(nullptr, tmp, d.vox_count.ptr, d.vox_start.ptr, (int)V + 1, st);
        RT_CUDA(ensure(d.cub_tmp, tmp));
        cub::DeviceScan::ExclusiveSum(d.cub_tmp.ptr, tmp, d.vox_count.ptr, d.vox_start.ptr, (int)V + 1, st);
        uint32_t R_h = 0;
        RT_CUDA(cudaMemcpyAsync(&R_h, d.vox_start.ptr + V, 4, cudaMemcpyDeviceToHost, st));
        trace.mark("vox count pass issued");
        RT_CUDA(cudaStreamSynchronize(st));
        trace.mark("sync 3 (reference count)");
        total_refs = R_h;
        RT_CUDA(ensure(d.vox_refs, (size_t)total_refs + 1));
        RT_CUDA(cudaMemsetAsync(d.vox_count.ptr, 0, ((size_t)V + 2) * 4, st));
        k_vox_pass<true><<<(n + tb - 1) / tb, tb, 0, st>>>(geom, d.sph_flag.ptr, n, grid, d.vox_count.ptr, d.vox_start.ptr, d.vox_refs.ptr);
        k_vox_finish<<<(V + tb - 1) / tb, tb, 0, st>>>(d.vox_start.ptr, V, d.vox_refs.ptr, d.vox.ptr);
        RT_CUDA(ensure(d.ref_geom, (size_t)total_refs + 4));   // (the cooperative kernel loads up to 3 entries past a list)
        if (total_refs)
            k_gather_geom<<<(unsigned)(((size_t)total_refs + tb - 1) / tb), tb, 0, st>>>(geom, d.vox_refs.ptr, total_refs, d.ref_geom.ptr);
    }
    RT_CUDA(d.prolog_geom.reserve(kMaxBig + 1));
    k_gather_geom<<<1, kMaxBig + 1, 0, st>>>(geom, d.big_refs.ptr, (size_t)(1 + nbig), d.prolog_geom.ptr);
    RT_CUDA(cudaGetLastError());
    grid.vox = d.vox.ptr;
    grid.refs = d.vox_refs.ptr;
    grid.ref_geom = d.ref_geom.ptr;
    built = true;
    n_spheres = n;
    trace.mark("fill passes issued (async)");
    return cudaSuccess;
}

size_t OctreeBuilder::reference_bytes(int spl_, bool fp16_) {
    return (size_t)kNumberNodes * (fp16_ ? kNodeBytesHalf : kNodeInts * 4) + (size_t)(kNumberLeafs + 1) * (size_t)(spl_ + 1) * 4 + 8;
}

cudaError_t OctreeBuilder::export_reference(cudaStream_t st, void *host_blob, size_t bytes) {
    if (!built) return cudaErrorNotReady;
    const size_t need = reference_bytes(spl, fp16);
    if (bytes < need) return cudaErrorInvalidValue;
    RT_CUDA(ensure(d.blob, need));
    RT_CUDA(cudaMemsetAsync(d.blob.ptr, 0, need, st));          // `new Octree()` value-initialises
    int *leaf_count = d.leaf_index.ptr + kCells * 8;
    RT_CUDA(cudaMemsetAsync(leaf_count, 0, 4, st));
    k_leaf_number<<<(kCells * 8 + 255) / 256, 256, 0, st>>>(d.vals_sorted.ptr, d.cell_start.ptr, spl, d.leaf_index.ptr, leaf_count);
    // the leaves follow the nodes: OctLeaf is all ints in both layouts, and the buckets of an FP16 build are its own memberships
    int32_t *leaves = reinterpret_cast<int32_t *>(d.blob.ptr + (size_t)kNumberNodes * (fp16 ? kNodeBytesHalf : kNodeInts * 4));
    if (fp16) k_blob_nodes<true><<<(kNumberNodes + 255) / 256, 256, 0, st>>>(d.node_of_potential.ptr, d.leaf_index.ptr, planes, d.blob.ptr);
    else k_blob_nodes<false><<<(kNumberNodes + 255) / 256, 256, 0, st>>>(d.node_of_potential.ptr, d.leaf_index.ptr, planes, d.blob.ptr);
    if (E > 0)
        k_blob_leaves<<<(E + 255) / 256, 256, 0, st>>>(d.keys_sorted.ptr, d.vals_sorted.ptr, d.cell_start.ptr, E, spl, d.leaf_index.ptr, leaves);
    int lc = 0;
    RT_CUDA(cudaMemcpyAsync(&lc, leaf_count, 4, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    leaf_count_h = lc + 1;                                   // leafCount starts at 1 (:60)
    const int32_t tail[2] = {counts.node_count, leaf_count_h};
    RT_CUDA(cudaMemcpyAsync(d.blob.ptr + need - 8, tail, 8, cudaMemcpyHostToDevice, st));
    RT_CUDA(cudaMemcpyAsync(host_blob, d.blob.ptr, need, cudaMemcpyDeviceToHost, st));
    RT_CUDA(cudaStreamSynchronize(st));
    blob_valid = true;
    return cudaGetLastError();
}

size_t OctreeBuilder::debug_read(cudaStream_t st, int which, void *host, size_t cap_bytes) const {
    if (!built) return 0;
    const void *src = nullptr;
    size_t bytes = 0;
    float desc[15];
    switch (which) {
        case 0:   // grid descriptor: org, hi, vs, inv_vs (12 floats) + nx, ny, nz (3 ints)
            for (int k = 0; k < 3; k++) { desc[k] = grid.org[k]; desc[3 + k] = grid.hi[k]; desc[6 + k] = grid.vs[k]; desc[9 + k] = grid.inv_vs[k]; }
            memcpy(desc + 12, &grid.nx, 4); memcpy(desc + 13, &grid.ny, 4); memcpy(desc + 14, &grid.nz, 4);
            if (host && cap_bytes >= sizeof desc) memcpy(host, desc, sizeof desc);
            return sizeof desc;
        case 1: src = d.vox.ptr; bytes = (size_t)total_voxels * sizeof(uint2); break;
        case 2: src = d.vox_refs.ptr; bytes = (size_t)total_refs * 4; break;
        case 3: src = d.ent_off.ptr; bytes = ((size_t)n_spheres + 1) * 4; break;
        case 4: src = d.ent_cell.ptr; bytes = (size_t)E * 2; break;
        case 5: src = d.big_refs.ptr + 1; bytes = (size_t)nbig * 4; break;
        case 6: src = d.sph_flag.ptr; bytes = (size_t)n_spheres; break;
        case 7: src = d.cell_start.ptr; bytes = (size_t)(kCells + 1) * 4; break;
        case 8: src = d.vals_sorted.ptr; bytes = (size_t)E * 4; break;
        default: return 0;
    }
    if (!host) return bytes;
    if (cap_bytes < bytes) return 0;
    if (bytes && cudaMemcpyAsync(host, src, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess) return 0;
    cudaStreamSynchronize(st);
    return bytes;
}

TreeView OctreeBuilder::view() const {
    TreeView v;
    memset(&v, 0, sizeof v);
    v.grid = grid;
    v.vis.ent_off = d.ent_off.ptr;
    v.vis.ent_cell = d.ent_cell.ptr;
    v.cell_list = d.vals_sorted.ptr;
    v.cell_start = d.cell_start.ptr;
    v.cell_cap = 8 * spl;
    v.check_visibility = all_spheres ? 0 : 1;
    v.prolog = d.big_refs.ptr;
    v.prolog_geom = d.prolog_geom.ptr;
    v.nprolog = 1 + nbig;
    v.slot0_none = slot0_none;
    for (int a = 0; a < 3; a++) for (int i = 0; i < kPlanes; i++) v.planes[a][i] = planes.p[a][i];
    v.no_drops = stats_h[1] == 0 ? 1 : 0;
    for (int a = 0; a < 3; a++) v.cell_inv[a] = 8.0f / (planes.p[a][kPlanes - 1] - planes.p[a][0]);
    return v;
}

}  // namespace rt
