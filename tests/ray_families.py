"""Ray families for the per-ray closest-hit tests (tests/test_closest_hit_rays_host.py on the host walks, tests/test_gpu_closest_hit_rays.py
on the device walks): rays at the edges of a 3D-DDA over the voxel grid, each family seeded and vectorised.

Every family takes the scene's spheres, the voxel grid the build makes for it (`Grid`, from hostsim's hs_grid_geometry) and a seed, and
returns (origins, directions) as float32 [R, 3].  Origins stay within kSceneReach (40) of the grid box's far corner: the voxel lists are
padded for origins that close to the spheres (rt_build.cuh sphere_pad, DESIGN §3), and origins beyond that reach are a documented limit,
not an input class these tests may hold the walks to."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

REACH = 40.0                                       # rt_build.cuh kSceneReach
PLANES_XZ = np.float32(-11.0) + np.float32(2.75) * np.arange(9, dtype=np.float32)     # the reference's level-3 cell planes
PLANES_Y = np.float32(0.25) * np.arange(9, dtype=np.float32)
SCALES = (1e-19, 1e-3, 1e3, 1e18)                  # |d| of the magnitude family (1e-19: dot(d, d) denormal; 1e18: b*b overflows)
LAYOUT_TAILS = (1, 17, 31)                         # lengths 32k + r: the cooperative hook's last warp is partial


@dataclass
class Grid:
    org: np.ndarray        # float32[3]
    vs: np.ndarray         # float32[3] voxel size
    hi: np.ndarray         # float32[3]
    dims: np.ndarray       # int[3]
    voxels: int = 0
    refs: int = 0          # references in the voxel lists

    def long_lists(self) -> bool:
        """The library's rule for four candidates per lane in the cooperative walk (rt_abi.cu select_walk)."""
        return self.voxels > 0 and self.refs // self.voxels >= 40

    def plane(self, axis: int, k) -> np.ndarray:
        """Voxel plane k along an axis, rounded as the walk computes it: org + (float)k * vs."""
        k = np.asarray(k, np.float32)
        return (self.org[axis] + k * self.vs[axis]).astype(np.float32)


def grid_geometry(hostsim, sph, blob, spl, use_octree, density=4.0) -> Grid:
    out = np.zeros(9, np.float32)
    dims = np.zeros(3, np.int32)
    counts = np.zeros(2, np.uint64)
    hostsim.hs_grid_geometry.restype = C.c_int
    rc = hostsim.hs_grid_geometry(C.c_void_p(sph.ctypes.data), len(sph), C.c_void_p(blob.ctypes.data) if blob is not None else None,
                                  spl, int(use_octree), C.c_float(density), C.c_void_p(out.ctypes.data), C.c_void_p(dims.ctypes.data),
                                  C.c_void_p(counts.ctypes.data))
    assert rc == 0 and (dims > 0).all(), (rc, dims)
    return Grid(out[0:3].copy(), out[3:6].copy(), out[6:9].copy(), dims, int(counts[0]), int(counts[1]))


HOST_WALKS = {"trace_tree": 0, "coop_eager": 1, "coop_lazy": 2}


def host_trace(hostsim, sph, blob, spl, use_octree, walk, org, dirs, density=4.0):
    """hs_trace_rays: the product's walk compiled for the host (HOST_WALKS) on the octree's grid or the flat-list grid.
    A failing ray of either test file replays here: host_trace(hostsim, sph, blob, spl, octree, walk, org[None], dir[None])."""
    org, dirs = _f32(org, dirs)
    idx = np.zeros(len(org), np.int32)
    t = np.zeros(len(org), np.float32)
    hostsim.hs_trace_rays.restype = C.c_int
    rc = hostsim.hs_trace_rays(C.c_void_p(sph.ctypes.data), len(sph), C.c_void_p(blob.ctypes.data) if blob is not None else None, spl,
                               int(use_octree), C.c_float(density), HOST_WALKS[walk], len(org), C.c_void_p(org.ctypes.data),
                               C.c_void_p(dirs.ctypes.data), C.c_void_p(idx.ctypes.data), C.c_void_p(t.ctypes.data))
    assert rc == 0
    return idx, t


def first_mismatch(want_i, want_t, got_i, got_t):
    """Index of the first ray whose sphere index differs, or whose t differs in its bits on a hit; None when all agree."""
    bad = (want_i != got_i) | ((want_i >= 0) & (want_t.view(np.uint32) != got_t.view(np.uint32)))
    k = np.flatnonzero(bad)
    return (int(k[0]), int(len(k))) if len(k) else None


def zero_component_on_cell_plane(org, dirs):
    """Documented limit of octree mode (DESIGN §3): a zero direction component with the origin's coordinate exactly on one of the
    reference's level-3 cell planes of that axis.  The reference's slab test divides 0 by 0 there, so whether a box passes depends on
    the tree level, and the library, which tests the level-3 cell alone, can accept a sphere the reference's descent never reaches."""
    out = np.zeros(len(org), bool)
    for a, planes in ((0, PLANES_XZ), (1, PLANES_Y), (2, PLANES_XZ)):
        out |= (dirs[:, a] == 0) & np.isin(org[:, a], planes)
    return out


def outside_contract(org, dirs, octree):
    return zero_component_on_cell_plane(org, dirs) if octree else np.zeros(len(org), bool)


def describe(family, walk, k, org, dirs, want, got):
    return (f"family {family}, walk {walk}, ray {k}: origin {org[k].tolist()} direction {dirs[k].tolist()} "
            f"(float32 bits {org[k].view(np.uint32).tolist()} {dirs[k].view(np.uint32).tolist()}): oracle {want}, walk {got}")


def _unit(v):
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _within_reach(org, g: Grid):
    far = np.maximum(np.abs(org - g.org.astype(np.float64)), np.abs(org - g.hi.astype(np.float64)))
    return np.linalg.norm(far, axis=1) <= REACH


def _inside(rng, g: Grid, R, grow=0.0):
    lo, hi = g.org.astype(np.float64) - grow, g.hi.astype(np.float64) + grow
    return lo + (hi - lo) * rng.random((R, 3))


def _f32(org, dirs):
    return np.ascontiguousarray(org, np.float32), np.ascontiguousarray(dirs, np.float32)


# ---- the families ---------------------------------------------------------------------------------------------------------------
def outside_in(sph, g: Grid, seed, R):
    """The grid-box clip (ray_box) and the first voxel: origins on shells from just outside the box out to the reach, aimed into it
    through every face, edge and corner, from below the ground too."""
    rng = np.random.default_rng(seed)
    c = 0.5 * (g.org.astype(np.float64) + g.hi.astype(np.float64))
    half = np.maximum(0.5 * (g.hi.astype(np.float64) - g.org.astype(np.float64)), 1e-6)
    orgs = []
    while sum(len(o) for o in orgs) < R:
        u = _unit(rng.normal(size=(2 * R, 3)))
        # toward the box's corners and edges as often as toward its faces
        snap = rng.random((2 * R, 3)) < 0.3
        u = _unit(np.where(snap, np.sign(u) * half, u))
        t_face = np.min(half / np.maximum(np.abs(u), 1e-30), axis=1)
        gap = 10.0 ** rng.uniform(-4, np.log10(REACH), 2 * R)
        o = c + u * (t_face + gap)[:, None]
        orgs.append(o[_within_reach(o, g)])
    org = np.concatenate(orgs)[:R]
    target = _inside(rng, g, R)
    return _f32(org, target - org)


def plane_locked(sph, g: Grid, seed, R):
    """Division by zero in the DDA set-up and ray_box: origins with one or two coordinates exactly on voxel planes, on the reference's
    cell planes or on the grid box's faces, with the matching direction components +0, -0 or +-1e-40 (the ray lies in a face or runs
    along an edge)."""
    rng = np.random.default_rng(seed)
    org = _inside(rng, g, R, grow=1.0)
    dirs = rng.normal(size=(R, 3))
    nlock = 1 + (rng.random(R) < 0.4)
    zero = np.array([0.0, -0.0, 1e-40, -1e-40], np.float32)
    org32 = org.astype(np.float32)
    dirs32 = dirs.astype(np.float32)
    for r in range(R):
        axes = rng.choice(3, nlock[r], replace=False)
        for a in axes:
            kind = rng.integers(3)
            if kind == 0:
                v = g.plane(a, rng.integers(0, g.dims[a] + 1))
            elif kind == 1:
                v = (PLANES_Y if a == 1 else PLANES_XZ)[rng.integers(9)]
            else:
                v = (g.org if rng.random() < 0.5 else g.hi)[a]
            org32[r, a] = v
            dirs32[r, a] = zero[rng.integers(4)]
        if nlock[r] == 2 and rng.random() < 0.5:        # along the edge from outside the box, into it
            free = 3 - axes.sum()
            side = rng.random() < 0.5
            org32[r, free] = (g.org[free] - rng.uniform(0.01, 5.0)) if side else (g.hi[free] + rng.uniform(0.01, 5.0))
            dirs32[r, free] = np.float32(1.0 if side else -1.0) * np.float32(rng.uniform(0.1, 2.0))
    return _f32(org32, dirs32)


def diagonal(sph, g: Grid, seed, R):
    """Ties of the DDA's step choice: origins at voxel corners, directions proportional to the voxel size per axis, so that
    tmx == tmy == tmz at every step; a third of them off by +-1 ulp per component."""
    rng = np.random.default_rng(seed)
    k = np.stack([rng.integers(-1, g.dims[a] + 2, R) for a in range(3)], 1)
    org = np.stack([g.plane(a, k[:, a]) for a in range(3)], 1)
    sign = np.where(rng.random((R, 3)) < 0.5, -1.0, 1.0)
    mult = rng.choice([1.0, 1.0, 2.0, 3.0], size=(R, 3))
    dirs = (sign * mult * g.vs.astype(np.float64) * rng.choice([0.5, 1.0, 7.0], size=(R, 1))).astype(np.float32)
    off = rng.random(R) < 1 / 3
    step = rng.integers(-1, 2, size=(R, 3))
    nudged = dirs.copy()
    for s, to in ((1, np.inf), (-1, -np.inf)):
        m = off[:, None] & (step == s)
        nudged[m] = np.nextafter(dirs[m], np.float32(to))
    return _f32(org, nudged)


def magnitude(sph, g: Grid, seed, R):
    """Approximate arithmetic at the ends of the float range: the rays of the three families above with |d| = 1e-19 (dot(d, d)
    subnormal, flushed by rcp_trav; components that become subnormal make the DDA hold that axis fixed), 1e-3, 1e3 and 1e18
    (b*b overflows; the reference gets NaN)."""
    parts = [fam(sph, g, seed + 7 * i, max(1, R // 12)) for i, fam in enumerate((outside_in, plane_locked, diagonal))]
    org = np.concatenate([p[0] for p in parts])
    d = np.concatenate([p[1] for p in parts]).astype(np.float64)
    n = np.linalg.norm(d, axis=1, keepdims=True)
    d = np.where(n > 0, d / np.where(n > 0, n, 1), d)
    outs = [(org, d * s) for s in SCALES]
    return _f32(np.concatenate([o for o, _ in outs]), np.concatenate([x for _, x in outs]))


def _small(sph):
    live = np.flatnonzero((sph["mat"] >= 0) & (np.arange(len(sph)) > 0) & (np.abs(sph["radius"]) < 2.0) & (np.abs(sph["radius"]) > 0))
    assert len(live) > 0
    return live


def _carpet(sph):
    """The spheres of the most common radius: create_world's carpet of small spheres on the ground, without its three big ones."""
    small = _small(sph)
    r = np.abs(sph["radius"][small])
    vals, counts = np.unique(r, return_counts=True)
    return small[r == vals[np.argmax(counts)]]


def grazing(sph, g: Grid, seed, R):
    """Near-tangent roots (the pre-filter's error bounds, maybe_hit / maybe_hit_ub): rays passing a sphere's centre at |r|(1 + k 2^-22),
    from 0.3 to 4 units before it and from above the ground, so that the targeted sphere is what most of them meet first."""
    rng = np.random.default_rng(seed)
    idx = rng.choice(_small(sph), R)
    c = np.stack([sph["cx"][idx], sph["cy"][idx], sph["cz"][idx]], 1).astype(np.float64)
    r = np.abs(sph["radius"][idx]).astype(np.float64)
    u = _unit(rng.normal(size=(R, 3)))
    w = _unit(np.cross(u, rng.normal(size=(R, 3))))
    k = rng.integers(-64, 65, R)
    tangent = c + w * (r * (1.0 + k * 2.0 ** -22))[:, None]
    back = rng.uniform(0.3, 4.0, R)[:, None]
    org = tangent - u * back
    flip = org[:, 1] < tangent[:, 1]                     # come down onto the sphere, not up through the ground
    u = np.where(flip[:, None], -u, u)
    org = tangent - u * back
    return _f32(org, u * rng.choice([1.0, 0.3, 3.0], R)[:, None])


def skimming(sph, g: Grid, seed, R):
    """The longest walks and the exit cap at its limit: horizontal rays through the whole grid at the height of a carpet sphere's top
    (cy + |r|) within a few ulp or a little below it, so that they touch that sphere and pass near-tangent over every carpet sphere
    of the same height on the way."""
    rng = np.random.default_rng(seed)
    idx = rng.choice(_carpet(sph), R)
    top = (sph["cy"][idx] + np.abs(sph["radius"][idx])).astype(np.float32)
    ulps = rng.integers(-3, 4, R)
    y = top.copy()
    for s in range(1, 4):
        y = np.where(ulps >= s, np.nextafter(y, np.float32(np.inf)), y)
        y = np.where(ulps <= -s, np.nextafter(y, np.float32(-np.inf)), y)
    below = rng.random(R) < 0.5
    y = np.where(below, (top - 10.0 ** rng.uniform(-6, -2, R)).astype(np.float32), y)
    ang = rng.uniform(0, 2 * np.pi, R)
    dxz = np.stack([np.cos(ang), np.sin(ang)], 1)
    p = np.stack([sph["cx"][idx], sph["cz"][idx]], 1).astype(np.float64)
    lo, hi = g.org[[0, 2]].astype(np.float64), g.hi[[0, 2]].astype(np.float64)
    # back along -dxz from the sphere's top to the grid box's side, and a little beyond
    back = np.where(dxz > 0, (p - lo) / np.maximum(dxz, 1e-12), (hi - p) / np.maximum(-dxz, 1e-12))
    oxz = p - dxz * (np.min(back, axis=1) + rng.uniform(0.01, 2.0, R))[:, None]
    org = np.stack([oxz[:, 0], np.zeros(R), oxz[:, 1]], 1).astype(np.float32)
    org[:, 1] = y
    dy = rng.choice(np.array([0.0, -0.0, 1e-40, -1e-7, 1e-7]), R)
    return _f32(org, np.stack([dxz[:, 0], dy, dxz[:, 1]], 1))


def exit_cap(sph, g: Grid, seed, R):
    """The cooperative walk's exit cap (RayMeta::t_out): hit points within 1e-4 of a voxel plane that cuts the sphere, so that the root
    sits at the edge of the voxel the cap offers it in."""
    rng = np.random.default_rng(seed)
    idx = rng.choice(_small(sph), 4 * R)
    c = np.stack([sph["cx"][idx], sph["cy"][idx], sph["cz"][idx]], 1).astype(np.float64)
    r = np.abs(sph["radius"][idx]).astype(np.float64)
    a = rng.integers(0, 3, 4 * R)
    ca = c[np.arange(4 * R), a]
    org_a, vs_a = g.org.astype(np.float64)[a], g.vs.astype(np.float64)[a]
    k = np.round((ca - org_a) / vs_a + rng.uniform(-1, 1, 4 * R))
    plane = org_a + k * vs_a
    p_a = plane + rng.uniform(-1e-4, 1e-4, 4 * R)
    keep = np.abs(p_a - ca) < 0.98 * r
    c, r, a, p_a, ca = c[keep][:R], r[keep][:R], a[keep][:R], p_a[keep][:R], ca[keep][:R]
    n = len(c)
    rho = np.sqrt(r * r - (p_a - ca) ** 2)
    ang = rng.uniform(0, 2 * np.pi, n)
    p = c.copy()
    p[np.arange(n), a] = p_a
    b1, b2 = (a + 1) % 3, (a + 2) % 3
    p[np.arange(n), b1] += rho * np.cos(ang)
    p[np.arange(n), b2] += rho * np.sin(ang)
    normal = (p - c) / r[:, None]
    v = _unit(rng.normal(size=(n, 3)))
    v = np.where((v * normal).sum(1, keepdims=True) < 0, -v, v)          # from the outer side of the surface point
    org = p + v * rng.uniform(0.05, 12.0, n)[:, None]
    return _f32(org, -v * rng.choice([1.0, 0.25], n)[:, None])


def on_and_in(sph, rng, idx, depths=(1.0, 0.5)):
    """Rays from the surfaces (|r| out from the centre) and from inside (|r| / 2) of the spheres idx, outwards, inwards and at random."""
    c = np.stack([sph["cx"][idx], sph["cy"][idx], sph["cz"][idx]], 1).astype(np.float64)
    r = np.abs(sph["radius"][idx]).astype(np.float64)[:, None]
    u = rng.normal(size=(len(idx), 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    org, dirs = [], []
    for depth in depths:
        o = c + depth * r * u
        for d in (u, -u, rng.normal(size=u.shape)):
            org.append(o)
            dirs.append(d)
    return np.concatenate(org).astype(np.float32), np.concatenate(dirs).astype(np.float32)


def on_inside(sph, g: Grid, seed, R):
    """Roots at or below kTMin and the second root: origins on, just inside, halfway in and at the centre of spheres, outward, inward
    and at random."""
    rng = np.random.default_rng(seed)
    per = 3 * 4
    idx = rng.choice(_small(sph), max(1, R // per))
    return on_and_in(sph, rng, idx, depths=(1.0, 1.0 - 2.0 ** -20, 0.5, 0.0))


FAMILIES = {"outside_in": outside_in, "plane_locked": plane_locked, "diagonal": diagonal, "magnitude": magnitude,
            "grazing": grazing, "skimming": skimming, "exit_cap": exit_cap, "on_inside": on_inside}


def layouts(R, seed):
    """Orders of a family's rays for the warp-cooperative hook: as generated, shuffled (every warp mixes misses, long walks and near
    hits), and prefixes of length 32k + r (a partial last warp).  -> [(name, index array)]"""
    rng = np.random.default_rng(seed)
    out = [("generated", np.arange(R)), ("shuffled", rng.permutation(R))]
    for r in LAYOUT_TAILS:
        n = 32 * max(0, (R - r) // 32) + r
        if 0 < n <= R:
            out.append((f"32k+{r}", np.arange(n)))
    return out
