// rt_octree.h — host-side handle of the GPU octree build (rt_octree.cu).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "rt_buffer.h"
#include "rt_types.h"

namespace rt {

struct BuildPlanes {
    float p[3][kPlanes];
};
struct BuildCounts {
    int node_count;
};
struct GridPrep {                 // k_grid_prep output: bounding box (order-preserving uint encoding), counts, big list
    uint32_t lo[3], hi[3];
    uint32_t live, nbig;
    uint32_t slot0_none;          // slot 0 is undefined (TreeView::slot0_none)
    uint32_t big[kMaxBig];
};

class OctreeBuilder {
public:
    OctreeBuilder();

    // replaces D2H(spheres) + buildOctree + H2D(Octree), main.cu:405-415
    // fp16: the USE_FP16 build of the reference (half-rounded scene, half arithmetic in `intersects`)
    // all_spheres: grid over EVERY defined sphere, wherever it lies (the flat-list mode's candidate set), not only over
    // the ones some octree cell stores
    cudaError_t build(cudaStream_t st, const float4 *geom, const int *tag, int n, int spl, float density, bool fp16 = false,
                      bool all_spheres = false);
    static size_t reference_bytes(int spl, bool fp16 = false);
    // the tree in the reference's own layout (acceleration_structure.h:23-61), assembled on the GPU on demand; a tree built
    // with fp16 comes out in the layout of the USE_FP16 build (48-byte nodes)
    cudaError_t export_reference(cudaStream_t st, void *host_blob, size_t bytes);
    TreeView view() const;
    // test hook: copy one internal array to the host (0 grid descriptor, 1 voxel records, 2 voxel references,
    // 3 per-sphere entry offsets, 4 per-sphere cell lists, 5 big list, 6 sphere flags); returns the byte size when
    // host == nullptr
    size_t debug_read(cudaStream_t st, int which, void *host, size_t cap) const;

    bool built = false, blob_valid = false, fp16 = false, all_spheres = false;
    float grid_flat, grid_wide;       // voxel shape in slab-shaped scenes (choose_grid; tuning knob RT_GRID_SHAPE="flat:wide[:min spheres]")
    uint32_t grid_flat_min;
    int spl = 0, n_spheres = 0, leaf_count_h = 0;
    int nbig = 0;
    int slot0_none = 0;               // TreeView::slot0_none of the last build
    uint32_t prolog_h[kMaxBig + 1];   // staging for the async upload (must outlive build())
    uint32_t E = 0, total_refs = 0, total_voxels = 0;
    GridView grid;
    BuildCounts counts{};
    unsigned long long stats_h[4] = {0, 0, 0, 0};   // stored entries, dropped_full, dropped_outside, -
    BuildPlanes planes;

private:
    struct {
        Buffer<uint32_t> ranges, ent_count, ent_off, keys, vals, keys_sorted, vals_sorted, cell_count, cell_start;
        Buffer<uint16_t> ent_cell;
        Buffer<uint8_t> sph_flag;
        Buffer<unsigned long long> stats;
        Buffer<int> node_of_potential;
        Buffer<BuildCounts> counts;
        Buffer<GridPrep> prep;
        Buffer<uint32_t> big_refs;
        Buffer<uint32_t> vox_count, vox_start, vox_refs;
        Buffer<float4> ref_geom, prolog_geom;
        Buffer<uint2> vox;
        Buffer<uint8_t> cub_tmp;
        Buffer<int> leaf_index;
        Buffer<uint8_t> blob;
    } d;
};

}  // namespace rt
