// rt_types.h — plain-data layouts shared by the host code, the build kernels and the render kernel.
#pragma once
#include <stdint.h>
#include <vector_types.h>

namespace rt {

// ---- reference Octree layout constants (acceleration_structure.h:11-15) ----
constexpr int kTreeHeight = 3;
constexpr int kNumberNodes = 585;         // 1 + 8 + 64 + 512
constexpr int kNumberLeafs = 4096;
constexpr int kNodeInts = 15;             // OctNode: level, AABB (6 floats), children[8]
constexpr int kNodeBytesHalf = 48;        // OctNode under USE_FP16: level, AABB (6 halves), children[8]
constexpr int kCells = 512;               // level-3 cells of the fixed 8x8x8 subdivision
constexpr int kPlanes = 9;                // slab planes per axis at level 3

// Camera as the render kernel consumes it (camera.h:51-58): 22 floats, kept in constant memory.
struct CameraData {
    float origin[3], lower_left_corner[3], horizontal[3], vertical[3], u[3], v[3], w[3];
    float lens_radius;
};

// ---- traversal structure (internal; NOT the reference layout) ------------------------------------------------
// The reference's result is  argmin t  over  {ground} U { spheres stored in a level-3 cell whose AABB the ray's
// infinite line crosses }  (acceleration_structure.h:226-342).  That is evaluated here as
//   (1) find candidate spheres with ONE uniform grid over all "small" spheres (3D-DDA, surface x voxel lists) plus
//       a short list of "big" spheres tested directly, and
//   (2) for a candidate that would become the closest hit, check the reference's visibility rule: does any cell
//       that STORES the sphere (i.e. was not dropped on bucket overflow) pass the line/AABB slab test?
// so the octree is never walked: only its per-sphere cell lists (VisView) and its slab planes are needed.
constexpr int kMaxBig = 64;                 // big spheres tested directly (beyond that they go into the grid)
constexpr float kBigRadiusFrac = 0.25f;     // big: radius > this x longest level-3 cell edge.  Measured: putting the RTIOW
                                            // r = 1 spheres into the grid stretches its box from the 0.2-high carpet to y = 2 and
                                            // costs 5x (49 voxel steps per ray through empty space) — they stay in the prolog list
constexpr uint16_t kEntDropped = 0x8000;    // VisView::ent_cell flag: entry dropped by the reference ("Leaf nodes full")

struct GridView {
    float org[3], hi[3];        // grid box
    float vs[3], inv_vs[3];     // voxel size and its reciprocal
    int nx, ny, nz;             // 0 = no grid
    const uint2 *vox;           // {first reference, reference count} per voxel
    const uint32_t *refs;       // sphere indices, ascending inside a voxel
    const float4 *ref_geom;     // geom[refs[k]] copied into list order: the render kernels stream candidates with ONE
                                // dependent load instead of two (16 B per reference; 96 MB at C3, 4.9 GB at C5)
};

struct VisView {
    const uint32_t *ent_off;    // n + 1 offsets: the cells sphere i was inserted into are ent_cell[ent_off[i] .. ent_off[i+1])
    const uint16_t *ent_cell;   // Morton id of the level-3 cell | kEntDropped
};

struct SceneView {
    const float4 *geom;     // {cx, cy, cz, radius} per sphere
    const float4 *matl;     // {albedo.xyz, param}
    const int *tag;         // RT_MAT_*
    int n;
};

struct TreeView {
    GridView grid;
    VisView vis;
    const uint32_t *prolog;     // first candidate list of every ray: the ground sphere (index 0, tested unconditionally by
    int nprolog;                // hitTree :322-332), then the big spheres in ascending order; nprolog = 1 + nbig
    const float4 *prolog_geom;  // their geometry in list order
    float planes[3][kPlanes];   // slab plane coordinates per axis (exact floats of the reference subdivision)
    // the reference's own cell lists (USE_FP16 path walks these): cell m (9-bit Morton id) was offered
    // cell_list[cell_start[m] .. cell_start[m+1]) in ascending sphere order and stored the first cell_cap = 8*SPL of them
    const uint32_t *cell_list;
    const uint32_t *cell_start;
    int cell_cap;
    // 1: hitTree semantics — a candidate counts only if a cell that stores it is crossed by the ray's line (VisView);
    // 0: hitable_list semantics — every sphere is a candidate (the grid then serves the flat-list mode, USE_OCTREE off)
    int check_visibility;
    // inputs of the cheap sufficient condition in front of the visibility rule (rt_trace.cuh visible_fast):
    int no_drops;               // 1: the build dropped no entry ("Leaf nodes full" never happened), so a cell stores every sphere
                                //    whose centre its r-expanded box contains
    float cell_inv[3];          // 8 / root box extent per axis: cell index guess from a coordinate
};

}  // namespace rt
