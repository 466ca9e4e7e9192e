"""CPU tier: worlds and cameras a caller builds (rt_scene_upload, rt_camera_set(desc), the drop-in classes), rendered by the PRODUCT's
per-lane device code compiled for the host (tests/hostsim) and held bit-for-bit to the oracle in device arithmetic, in octree mode and
in the flat-list mode's grid (hitable_list::hit answered through the voxel lists, as the library does from 256 spheres on).

create_world's carpet of equal spheres never exercises what the traversal assumes about its input: hollow spheres (negative radius,
the RTIOW "hollow glass" idiom), exact duplicates (a tie on every hit), more big spheres than the prolog holds, centres on the cell
planes, degenerate radii, non-slab clouds, undefined slots.  The worlds here do; tests/test_gpu_caller_worlds.py renders the same
worlds and cameras on the GPU.  Cameras stay within kSceneReach (40) of the spheres, the reach the voxel padding is sized for."""
import ctypes as C

import numpy as np
import pytest

SPHERE_DTYPE = np.dtype(
    [("cx", "<f4"), ("cy", "<f4"), ("cz", "<f4"), ("radius", "<f4"), ("mat", "<i4"),
     ("ax", "<f4"), ("ay", "<f4"), ("az", "<f4"), ("param", "<f4")]
)
NONE, LAMBERTIAN, METAL, DIELECTRIC = -1, 0, 1, 2
MAX_BIG = 64                      # rt_types.h kMaxBig
BIG_RADIUS = 0.25 * 2.75          # kBigRadiusFrac x the longest level-3 cell edge
PLANES_XZ = [-11.0 + 2.75 * k for k in range(9)]
PLANES_Y = [0.25 * k for k in range(9)]


# ---- worlds ---------------------------------------------------------------------------------------------------------------------
def _material(rng):
    mat = int(rng.choice([LAMBERTIAN, METAL, DIELECTRIC], p=[0.5, 0.25, 0.25]))
    param = 1.5 if mat == DIELECTRIC else (0.5 * rng.random() if mat == METAL else 0.0)
    return (mat, rng.random(), rng.random(), rng.random(), param)


def _sphere(c, r, m):
    return (c[0], c[1], c[2], r) + tuple(m)


def _ground():
    return _sphere((0.0, -1000.0, 0.0), 1000.0, (LAMBERTIAN, 0.5, 0.5, 0.5, 0.0))


GLASS = (DIELECTRIC, 0.0, 0.0, 0.0, 1.5)
LANDMARK = (0.0, 1.0, 0.0)        # a glass sphere of radius 1 in every world: the "in_glass" camera sits inside it


def _carpet(rng, n):
    """Ground, the glass landmark, then spheres of radius 0.2 resting on the ground at random places."""
    out = [_ground(), _sphere(LANDMARK, 1.0, GLASS)]
    while len(out) < n:
        out.append(_sphere((rng.uniform(-11, 11), 0.2, rng.uniform(-11, 11)), 0.2, _material(rng)))
    return out


def _array(rows):
    a = np.zeros(len(rows), dtype=SPHERE_DTYPE)
    for i, r in enumerate(rows):
        a[i] = r
    return a


def world_hollow(n=1500, seed=1):
    """Hollow glass: (c, r) and (c, -0.9 r) or (c, -0.3 r), r in {0.2, 0.5, 1.0}; the landmark is one (the camera is in its hollow)."""
    rng = np.random.default_rng(seed)
    rows = [_ground(), _sphere(LANDMARK, 1.0, GLASS), _sphere(LANDMARK, -0.9, GLASS)]
    while len(rows) + 2 <= n:
        if rng.random() < 0.4:
            rows.append(_sphere((rng.uniform(-11, 11), 0.2, rng.uniform(-11, 11)), 0.2, _material(rng)))
            continue
        r = float(rng.choice([0.2, 0.5, 1.0]))
        c = (rng.uniform(-10.5, 10.5), r, rng.uniform(-10.5, 10.5))
        inner = float(rng.choice([-0.9, -0.3])) * r
        rows += [_sphere(c, r, GLASS), _sphere(c, inner, GLASS if rng.random() < 0.8 else _material(rng))]
    return _array(rows)


def world_duplicates(n=1500, seed=2):
    """The second half repeats the first half's spheres exactly, with other materials: every hit is an exact tie."""
    rng = np.random.default_rng(seed)
    first = _carpet(rng, (n + 1) // 2)
    rows = list(first)
    for r in first[1:]:
        if len(rows) >= n:
            break
        rows.append(r[:4] + _material(rng))
    return _array(rows)


def world_many_big(n=1500, seed=3):
    """More than kMaxBig big spheres (radius above a quarter cell edge): the prolog takes 64, the rest go into the grid."""
    rng = np.random.default_rng(seed)
    rows = _carpet(rng, n - 100)
    for _ in range(100):
        r = float(rng.uniform(0.7, 1.3))
        rows.append(_sphere((rng.uniform(-10, 10), rng.uniform(0.0, 2.0), rng.uniform(-10, 10)), r, _material(rng)))
    assert sum(r[3] > BIG_RADIUS for r in rows[1:]) > MAX_BIG
    return _array(rows)


def world_planes(n=1500, seed=4):
    """Centres on the level-3 cell planes (x, z multiples of 2.75 from -11, y multiples of 0.25) — on the root box's outer faces
    too — with radii that make surfaces touch the planes and each other."""
    rng = np.random.default_rng(seed)
    rows = [_ground(), _sphere(LANDMARK, 1.0, GLASS)]
    while len(rows) < n:
        c = (float(rng.choice(PLANES_XZ)), float(rng.choice(PLANES_Y)), float(rng.choice(PLANES_XZ)))
        r = float(rng.choice([0.05, 0.125, 0.25, 0.5, 0.6875, 1.375]))
        rows.append(_sphere(c, r, _material(rng)))
    return _array(rows)


def world_tiny(n=1500, seed=5):
    """Radii 1e-4 and 0 with real materials among the carpet."""
    rng = np.random.default_rng(seed)
    rows = _carpet(rng, n)
    for i in range(2, n):
        if rng.random() < 0.3:
            c = (rng.uniform(-11, 11), rng.uniform(0.0, 2.0), rng.uniform(-11, 11))
            rows[i] = _sphere(c, float(rng.choice([1e-4, 0.0])), _material(rng))
    return _array(rows)


def world_cloud(n=1500, seed=6, half=6.0, height=9.0):
    """A 3-D cloud, not a slab (cubic voxels, no flat-voxel rule); most of it lies above the octree's root box (y > 2)."""
    rng = np.random.default_rng(seed)
    rows = [_ground(), _sphere(LANDMARK, 1.0, GLASS)]
    while len(rows) < n:
        r = float(rng.choice([0.1, 0.2, 0.4], p=[0.5, 0.4, 0.1]))
        rows.append(_sphere((rng.uniform(-half, half), rng.uniform(0.2, height), rng.uniform(-half, half)), r, _material(rng)))
    return _array(rows)


def world_undefined(n=1500, seed=7):
    """Undefined slots (RT_MAT_NONE: never hit), slot 0 — the ground's geometry — among them."""
    rng = np.random.default_rng(seed)
    a = _array(_carpet(rng, n))
    a["mat"][0] = NONE
    a["mat"][rng.choice(np.arange(2, n), n // 20, replace=False)] = NONE
    return a


def world_dense(n=4000, seed=8):
    """Heavily overlapping spheres in a small cube: long voxel lists (>= 40 references per voxel)."""
    rng = np.random.default_rng(seed)
    rows = [_ground(), _sphere(LANDMARK, 1.0, GLASS)]
    while len(rows) < n:
        rows.append(_sphere((rng.uniform(-2, 2), rng.uniform(0.6, 4.6), rng.uniform(-2, 2)), 0.65, _material(rng)))
    return _array(rows)


WORLDS = {"hollow": world_hollow, "duplicates": world_duplicates, "many_big": world_many_big, "planes": world_planes,
          "tiny": world_tiny, "cloud": world_cloud, "undefined": world_undefined}


# ---- cameras --------------------------------------------------------------------------------------------------------------------
CAMERAS = {
    "low": dict(lookfrom=(3.0, 0.45, 2.2), lookat=(-4.0, 0.3, -1.0), vup=(0.0, 1.0, 0.0), vfov=55.0, aperture=0.0, focus_dist=6.0),
    "topdown": dict(lookfrom=(0.7, 16.0, -0.4), lookat=(0.0, 0.0, 0.0), vup=(0.0, 0.0, 1.0), vfov=70.0, aperture=0.1, focus_dist=16.0),
    "wide_aperture": dict(lookfrom=(12.0, 2.5, 4.0), lookat=(0.0, 0.5, 0.0), vup=(0.0, 1.0, 0.0), vfov=30.0, aperture=2.0,
                          focus_dist=11.0),
    "in_glass": dict(lookfrom=(0.1, 1.05, 0.05), lookat=(-5.0, 0.6, -3.0), vup=(0.0, 1.0, 0.0), vfov=75.0, aperture=0.0,
                     focus_dist=5.0),
}


def camera22(desc, aspect):
    """camera.h:22-44 in float64: origin, lower_left_corner, horizontal, vertical, u, v, w, lens_radius (22 values)."""
    lookfrom, lookat, vup = (np.asarray(desc[k], np.float64) for k in ("lookfrom", "lookat", "vup"))
    theta = desc["vfov"] * np.pi / 180.0
    half_height = np.tan(theta / 2.0)
    half_width = aspect * half_height
    f = desc["focus_dist"]
    w = (lookfrom - lookat) / np.linalg.norm(lookfrom - lookat)
    u = np.cross(vup, w)
    u /= np.linalg.norm(u)
    v = np.cross(w, u)
    llc = lookfrom - half_width * f * u - half_height * f * v - f * w
    return np.concatenate([lookfrom, llc, 2 * half_width * f * u, 2 * half_height * f * v, u, v, w, [desc["aperture"] / 2.0]])


# ---- host renders ---------------------------------------------------------------------------------------------------------------
SPL = 30


def _render_both(hostsim, O, sph, cam, nx, ny, ns, octree):
    """(product frame, oracle frame, product rays, oracle rays, coop rays, coop mismatches, grid voxels, grid references)"""
    blob = O.build_octree(sph, SPL)[0] if octree else None
    p = O.make_params(nx, ny, ns, octree, SPL, O.ARITH_DEVICE)
    ref, _, ctr = O.render(sph, O.Camera.from_buffer_copy(cam.tobytes()), p, blob)
    fb = np.zeros((ny, nx, 3), np.float32)
    c = O.Counters()
    stats = np.zeros(2, np.uint64)
    hostsim.hs_set_list_grid(0 if octree else 1)
    hostsim.hs_coop_check(1)
    try:
        hostsim.hs_render(C.c_void_p(sph.ctypes.data), len(sph), C.c_void_p(cam.ctypes.data),
                          C.c_void_p(blob.ctypes.data) if blob is not None else None, C.byref(p), C.c_float(4.0),
                          C.c_void_p(fb.ctypes.data), None, C.byref(c), C.c_void_p(stats.ctypes.data))
        rays, bad = C.c_ulonglong(0), C.c_ulonglong(0)
        hostsim.hs_coop_check_result(C.byref(rays), C.byref(bad))
    finally:
        hostsim.hs_coop_check(0)
        hostsim.hs_set_list_grid(0)
    return fb, ref, int(c.rays), int(ctr["rays"]), rays.value, bad.value, int(stats[0]), int(stats[1])


@pytest.mark.parametrize("octree", [True, False], ids=["octree", "list_grid"])
@pytest.mark.parametrize("world", list(WORLDS))
def test_caller_world_matches_oracle(hostsim, O, world, octree):
    """Every camera: bit-identical frame, equal ray count, and the cooperative kernel's candidate rule returns trace_walk's
    minimum on every ray (host emulation, both extreme schedules)."""
    sph = WORLDS[world]()
    nx, ny, ns = 64, 48, 2
    for name, desc in CAMERAS.items():
        cam = camera22(desc, nx / ny).astype(np.float32)
        fb, ref, rays, ref_rays, coop_rays, coop_bad, voxels, _ = _render_both(hostsim, O, sph, cam, nx, ny, ns, octree)
        assert voxels > 0
        same = (fb.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
        assert same.all(), f"{name}: {int((~same).sum())} of {nx * ny} pixels differ from the oracle"
        assert rays == ref_rays, name
        assert coop_rays == rays and coop_bad == 0, (name, coop_rays, coop_bad)


def test_dense_list_world_has_long_voxel_lists(hostsim, O):
    """The world that sends the cooperative kernel to four candidates per lane (>= 40 references per voxel) renders the oracle's frame."""
    sph = world_dense()
    nx, ny, ns = 48, 32, 2
    cam = camera22(CAMERAS["wide_aperture"], nx / ny).astype(np.float32)
    fb, ref, rays, ref_rays, coop_rays, coop_bad, voxels, refs = _render_both(hostsim, O, sph, cam, nx, ny, ns, False)
    assert refs // voxels >= 40, (voxels, refs)
    assert np.array_equal(fb.view(np.uint32), ref.view(np.uint32)) and rays == ref_rays
    assert coop_rays == rays and coop_bad == 0


def test_hollow_spheres_are_hit_through_the_list_grid(hostsim, O):
    """The grid lists a hollow sphere's surface at |r|: a ray from the camera in the landmark's hollow reaches the sky only through
    the inner (r = -0.9) and outer (r = 1) surfaces, so a frame without them differs from the oracle on every pixel."""
    sph = world_hollow()
    nx, ny = 32, 24
    cam = camera22(CAMERAS["in_glass"], nx / ny).astype(np.float32)
    fb, ref, rays, ref_rays, *_ = _render_both(hostsim, O, sph, cam, nx, ny, 1, False)
    assert np.array_equal(fb.view(np.uint32), ref.view(np.uint32)) and rays == ref_rays
    assert ref_rays >= 3 * nx * ny                # every path crosses the two surfaces before it leaves (at least 3 segments)


def test_undefined_slot_zero_is_never_hit(hostsim, O):
    """RT_MAT_NONE marks a slot that is never hit, slot 0 included, in octree mode as in the flat list: a downward camera sees
    no ground, and the two modes agree wherever the frame does not depend on the octree's visibility rule."""
    sph = world_undefined()
    nx, ny = 48, 32
    cam = camera22(CAMERAS["topdown"], nx / ny).astype(np.float32)
    fb_o, ref_o, rays_o, ref_rays_o, *_ = _render_both(hostsim, O, sph, cam, nx, ny, 1, True)
    assert np.array_equal(fb_o.view(np.uint32), ref_o.view(np.uint32)) and rays_o == ref_rays_o
    with_ground = sph.copy()
    with_ground["mat"][0] = LAMBERTIAN
    fb_g, _, rays_g, *_ = _render_both(hostsim, O, with_ground, cam, nx, ny, 1, True)
    assert rays_o < rays_g                        # without slot 0 the rays that would hit the ground go to the sky
