"""GPU tier (-m gpu): caller-built worlds (rt.upload_world) and cameras (rt.set_camera with a CameraDesc) through every FP32 render
kernel, against the oracle.  The worlds and cameras are tests/test_caller_worlds_host.py's, where the product's device code, compiled
for the host, renders them bit-identical to the oracle; here the CUDA kernels must do the same at test_gpu_parity's bar.

The oracle renders with the camera read back from the library (rt.camera()), so the frames check the render; the camera constructor
itself is checked against a float64 restatement of camera.h (a wrong sign there would otherwise go unnoticed: the oracle would inherit it)."""
import ctypes as C

import numpy as np
import pytest

import ray_families as F
import test_caller_worlds_host as W

pytestmark = pytest.mark.gpu

POWF_ALLOWANCE = 1e-4             # libdevice powf (schlick) against libm powf, as in test_gpu_parity
SPL = 30
KERNEL_LANE, KERNEL_COOP, KERNEL_SWEEP = "k_render<octree>", "k_render_coop", "k_render<list>"
# variants: 0 the automatic choice, 1 the per-lane grid walk, 40 the warp-cooperative kernel, 20 the N-test sweep (flat list only)
VARIANTS = {True: (0, 1, 40), False: (0, 1, 40, 20)}


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


def _desc(pkg, d, aspect):
    f3 = C.c_float * 3
    return pkg.CameraDesc(f3(*d["lookfrom"]), f3(*d["lookat"]), f3(*d["vup"]), d["vfov"], aspect, d["aperture"], d["focus_dist"])


def _upload(rt, O, sph, octree):
    rt.upload_world(sph)
    if not octree:
        return None
    rt.build_octree(SPL)
    blob, _ = O.build_octree(sph, SPL)
    assert rt.export_octree().tobytes() == blob.tobytes()
    return blob


def _check_frames(rt, pkg, O, sph, blob, octree, cameras, nx, ny, ns, variants, expect_auto=None, spl=SPL, stride=1, **kw):
    """Every camera through every variant: >= 1 - POWF_ALLOWANCE of the pixels (over all cameras) bit-identical to the oracle, rays
    within the same allowance, and every variant's frame bit-identical to the first variant's (all kernels share libdevice).
    stride > 1: the oracle renders every stride-th pixel of every stride-th row, and the rays of those pixels come from
    rt.render_pixels (a pixel list computes exactly the frame's pixels)."""
    seed_mode = kw.get("seed_mode", pkg.SEED_HEAD)
    sub = (slice(None, None, stride), slice(None, None, stride))
    pix = (np.arange(0, ny, stride)[:, None] * nx + np.arange(0, nx, stride)[None, :]).astype(np.uint32).ravel()
    bad = {v: 0 for v in variants}          # pixels that differ from the oracle
    apart = {v: 0 for v in variants}        # pixels that differ from the first variant's frame
    rays = {v: 0 for v in variants}
    ref_rays = pixels = 0
    for name in cameras:
        rt.set_camera(nx, ny, _desc(pkg, W.CAMERAS[name], nx / ny))
        cam = O.Camera.from_buffer_copy(rt.camera().tobytes())
        ref, _, ctr = O.render(sph, cam, O.make_params(nx, ny, ns, octree, spl, O.ARITH_DEVICE, step=(stride, stride), seed_mode=seed_mode),
                               blob)
        first = None
        for v in variants:
            fb, s = rt.render(nx, ny, ns, use_octree=octree, variant=v, **kw)
            want = {0: expect_auto, 40: KERNEL_COOP, 20: KERNEL_SWEEP}.get(v)
            assert want is None or s["kernel"].startswith(want), (v, s["kernel"])
            assert s["paths"] == nx * ny * ns
            first = fb if first is None else first
            apart[v] += int((fb.view(np.uint32) != first.view(np.uint32)).any(axis=2).sum())
            bad[v] += int((fb[sub].view(np.uint32) != ref[sub].view(np.uint32)).any(axis=2).sum())
            if stride > 1:
                s = rt.render_pixels(nx, ny, ns, pix, use_octree=octree, variant=v, **kw)[1]
            rays[v] += int(s["rays"])
        ref_rays += ctr["rays"]
        pixels += len(pix)
    report = {v: dict(differ_from_oracle=bad[v], differ_from_first=apart[v], rays=rays[v]) for v in variants}
    msg = f"{pixels} pixels, oracle rays {ref_rays}: {report}"
    assert all(apart[v] == 0 for v in variants), msg
    assert all(bad[v] <= POWF_ALLOWANCE * pixels for v in variants), msg
    assert all(abs(rays[v] - ref_rays) <= max(2, int(POWF_ALLOWANCE * ref_rays)) for v in variants), msg


@pytest.mark.parametrize("octree", [True, False], ids=["octree", "list"])
@pytest.mark.parametrize("world", list(W.WORLDS))
def test_caller_world_kernels_match_oracle(rt, pkg, O, world, octree):
    sph = W.WORLDS[world]()
    blob = _upload(rt, O, sph, octree)
    _check_frames(rt, pkg, O, sph, blob, octree, list(W.CAMERAS), 80, 48, 2, VARIANTS[octree], expect_auto=KERNEL_LANE)


def _inject_hollow_and_duplicates(sph, rng, count):
    """Append a hollow inner sphere (-0.9 r or -0.3 r) for `count` spheres and an exact duplicate, with another material, of `count` more."""
    live = np.flatnonzero(sph["mat"][1:] >= 0) + 1
    pick = rng.choice(live, 2 * count, replace=False)
    inner = sph[pick[:count]].copy()
    inner["radius"] *= rng.choice(np.array([-0.9, -0.3], np.float32), count)
    inner["mat"] = W.DIELECTRIC
    inner["param"] = 1.5
    dup = sph[pick[count:]].copy()
    dup["mat"] = (dup["mat"] + 1) % 3
    dup["param"] = np.where(dup["mat"] == W.DIELECTRIC, 1.5, 0.3).astype(np.float32)
    return np.concatenate([sph, inner, dup])


def test_large_octree_world_with_hollow_spheres_and_duplicates(rt, pkg, O):
    """create_world(100000) with 3 000 hollow inner spheres and 3 000 exact duplicates: the automatic choice is the cooperative kernel."""
    sph = _inject_hollow_and_duplicates(O.create_world(100000)[0], np.random.default_rng(21), 3000)
    rt.upload_world(sph)
    rt.build_octree(300)
    blob, _ = O.build_octree(sph, 300)
    _check_frames(rt, pkg, O, sph, blob, True, ["low", "wide_aperture"], 160, 96, 2, VARIANTS[True], expect_auto=KERNEL_COOP, spl=300)


def test_large_list_cloud(rt, pkg, O):
    """A 60 000-sphere 3-D cloud in flat-list mode: cubic voxels, no slab rule, the cooperative kernel by the automatic choice."""
    sph = W.world_cloud(60000, seed=22, half=8.0, height=16.0)
    rt.upload_world(sph)
    _check_frames(rt, pkg, O, sph, None, False, ["low", "topdown"], 96, 64, 1, VARIANTS[False], expect_auto=KERNEL_COOP, stride=4)


def test_dense_list_world_four_candidates_per_lane(rt, pkg, O):
    """>= 40 references per voxel (checked on the same build rules by the CPU tier): the cooperative kernel takes four candidates per
    lane and chunk step."""
    sph = W.world_dense()
    rt.upload_world(sph)
    _check_frames(rt, pkg, O, sph, None, False, ["wide_aperture", "in_glass"], 64, 48, 2, (40, 1, 20))


@pytest.mark.parametrize("octree", [True, False], ids=["octree", "list"])
@pytest.mark.parametrize("world", ["hollow", "duplicates"])
def test_closest_hit_from_on_and_inside_spheres(rt, O, world, octree):
    """rt.trace_rays against O.closest_hit: index and t bit-identical.  Ties between duplicates: the lower index in the flat list,
    the reference's cell order (tie_key) in the octree."""
    sph = W.WORLDS[world]()
    blob = _upload(rt, O, sph, octree)
    rng = np.random.default_rng(31)
    if world == "hollow":
        idx = np.flatnonzero(sph["radius"] < 0)
        idx = np.concatenate([idx, idx - 1])                       # the inner spheres and their outer shells
    else:
        idx = rng.choice(np.arange(len(sph) // 2 + 1, len(sph)), 150, replace=False)    # the duplicates
    idx = rng.choice(idx, min(len(idx), 150), replace=False)
    org, dirs = F.on_and_in(sph, rng, idx)
    gi, gt = rt.trace_rays(org, dirs, octree)
    hits = 0
    for k in range(len(org)):
        oi, ot = O.closest_hit(sph, org[k], dirs[k], blob, SPL, octree)
        assert oi == gi[k] and (oi < 0 or np.float32(ot) == gt[k]), (k, oi, ot, gi[k], gt[k])
        hits += oi > 0
    assert hits > len(org) // 4


def test_upstream_seeding_on_a_caller_world(rt, pkg, O):
    sph = W.world_hollow()
    _upload(rt, O, sph, False)
    _check_frames(rt, pkg, O, sph, None, False, ["in_glass", "wide_aperture"], 64, 48, 2, (0, 40), seed_mode=pkg.SEED_UPSTREAM)


def test_render_pixels_on_a_caller_world(rt, pkg, O):
    """A window of a caller world's frame through rt.render_pixels is the frame's pixels, bit for bit, with a custom camera."""
    sph = W.world_duplicates()
    blob = _upload(rt, O, sph, True)
    nx, ny, ns = 80, 48, 2
    rt.set_camera(nx, ny, _desc(pkg, W.CAMERAS["low"], nx / ny))
    for v in (1, 40):
        fb, _ = rt.render(nx, ny, ns, use_octree=True, variant=v)
        i0, i1, j0, j1 = 13, 61, 5, 37
        vals, _ = rt.render_pixels(nx, ny, ns, pkg.window_pixels(nx, ny, i0, i1, j0, j1), use_octree=True, variant=v)
        win = np.zeros((j1 - j0, i1 - i0, 3), np.float32)
        pix = pkg.window_pixels(nx, ny, i0, i1, j0, j1).astype(np.int64)
        win[pix // nx - j0, pix % nx - i0] = vals
        assert np.array_equal(win.view(np.uint32), fb[j0:j1, i0:i1].view(np.uint32)), v
    ref, _, _ = O.render(sph, O.Camera.from_buffer_copy(rt.camera().tobytes()), O.make_params(nx, ny, ns, True, SPL, O.ARITH_DEVICE), blob)
    assert (fb.view(np.uint32) == ref.view(np.uint32)).all(axis=2).mean() >= 1 - POWF_ALLOWANCE


@pytest.mark.parametrize("name,aspect", [("low", 1.5), ("topdown", 0.75), ("wide_aperture", 16 / 9), ("in_glass", 2.0)])
def test_camera_from_a_description(rt, pkg, name, aspect):
    """k_camera_setup against camera.h:22-44 in float64 (not a bit test: the reference never builds a runtime camera)."""
    rt.create_world(8, 0.1)
    desc = W.CAMERAS[name]
    rt.set_camera(120, 80, _desc(pkg, desc, aspect))          # the description's aspect ratio is kept, whatever the frame size
    got = rt.camera().astype(np.float64)
    want = W.camera22(desc, aspect)
    for k in range(7):                                        # per 3-vector, relative to its length
        g, w = got[3 * k:3 * k + 3], want[3 * k:3 * k + 3]
        assert np.abs(g - w).max() <= 1e-5 * max(1.0, np.linalg.norm(w)), (name, k, g, w)
    assert got[21] == np.float32(desc["aperture"] / 2)
    assert np.dot(got[12:15], got[15:18]) == pytest.approx(0, abs=1e-6)      # u, v, w orthonormal, right-handed (w = u x v)
    assert np.allclose(np.cross(got[12:15], got[15:18]), got[18:21], atol=1e-6)
