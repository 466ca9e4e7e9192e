"""CPU tier: the product's closest-hit walks (rt_trace.cuh trace_tree, and the cooperative walk's candidate rule under both extreme
schedules followed by finish_hit), compiled for the host by tests/hostsim, ray by ray against the oracle in device arithmetic, on the
ray families of tests/ray_families.py — the inputs where a 3D-DDA goes wrong.  Octree mode on create_world scenes (20 000 / 30
overflows leaf buckets: the sphere_visible path), and the flat-list mode's grid over all spheres.

The host walks evaluate one ray at a time with exact 1/x and sqrtf (rt_trace.cuh rcp_trav / sqrt_trav), so the warp layouts and the
approximate arithmetic are left to tests/test_gpu_closest_hit_rays.py; here a mismatch means the walk's logic is wrong."""
import numpy as np
import pytest

import ray_families as F

RAYS = 2000                     # per family and scene

SCENES = {                      # name: (spheres, spl, octree)
    "oct488": (488, 30, True),
    "oct8000": (8000, 30, True),
    "oct20000": (20000, 30, True),
    "oct100000": (100000, 300, True),
    "list488": (488, 30, False),
    "list6000": (6000, 30, False),
}


@pytest.mark.parametrize("scene", list(SCENES))
def test_every_host_walk_matches_the_oracle_on_every_family(hostsim, O, scene):
    n, spl, octree = SCENES[scene]
    sph, _ = O.create_world(n)
    blob = O.build_octree(sph, spl)[0] if octree else None
    g = F.grid_geometry(hostsim, sph, blob, spl, octree)
    report = {}
    for fi, (family, make) in enumerate(F.FAMILIES.items()):
        org, dirs = make(sph, g, 1000 * n + fi, RAYS)
        keep = ~F.outside_contract(org, dirs, octree)        # (test_documented_limits_still_differ holds those to their description)
        org, dirs = org[keep], dirs[keep]
        want_i, want_t = O.closest_hits(sph, org, dirs, blob, spl, octree)
        hits = int((want_i >= 0).sum())
        assert (want_i > 0).any(), f"family {family} hits no sphere but the ground in {scene}"
        for walk in F.HOST_WALKS:
            got_i, got_t = F.host_trace(hostsim, sph, blob, spl, octree, walk, org, dirs)
            bad = F.first_mismatch(want_i, want_t, got_i, got_t)
            assert bad is None, f"{scene}: {bad[1]} rays differ; " + F.describe(
                family, walk, bad[0], org, dirs, (int(want_i[bad[0]]), float(want_t[bad[0]])), (int(got_i[bad[0]]), float(got_t[bad[0]])))
        report[family] = (len(org), hits, int((~keep).sum()))
    print(scene, "family: (rays, oracle hits, rays outside the contract)", report)


@pytest.mark.xfail(strict=True, reason="documented input class (DESIGN §3): the octree walks may answer it unlike the reference")
def test_zero_component_on_a_cell_plane_still_differs(hostsim, O):
    """The plane-locked family's rays of the one documented class, which the bar above leaves out, through trace_tree: some differ
    from the oracle today.  The day a fix makes them agree this test passes, fails as a strict xfail, and the class leaves the contract."""
    n, spl, octree = SCENES["oct100000"]
    sph, _ = O.create_world(n)
    blob = O.build_octree(sph, spl)[0] if octree else None
    g = F.grid_geometry(hostsim, sph, blob, spl, octree)
    org, dirs = F.plane_locked(sph, g, 1000 * n + list(F.FAMILIES).index("plane_locked"), RAYS)
    sel = F.zero_component_on_cell_plane(org, dirs)
    org, dirs = org[sel], dirs[sel]
    want_i, want_t = O.closest_hits(sph, org, dirs, blob, spl, octree)
    got_i, got_t = F.host_trace(hostsim, sph, blob, spl, octree, "trace_tree", org, dirs)
    assert F.first_mismatch(want_i, want_t, got_i, got_t) is None


def test_batched_oracle_is_the_single_ray_query(O):
    """rto_closest_hits is rto_closest_hit in a loop over the rays (OpenMP), in both modes."""
    sph, _ = O.create_world(488)
    blob, _ = O.build_octree(sph, 30)
    rng = np.random.default_rng(3)
    R = 300
    org = np.stack([rng.uniform(-13, 14, R), rng.uniform(-0.5, 3, R), rng.uniform(-13, 13, R)], 1).astype(np.float32)
    dirs = rng.normal(size=(R, 3)).astype(np.float32)
    dirs[:30, 1] = 0.0
    for octree in (True, False):
        bi, bt = O.closest_hits(sph, org, dirs, blob, 30, octree)
        hits = 0
        for k in range(R):
            oi, ot = O.closest_hit(sph, org[k], dirs[k], blob, 30, octree)
            assert oi == bi[k] and np.float32(ot).view(np.uint32) == bt[k].view(np.uint32), (octree, k)
            hits += oi >= 0
        assert 0 < hits < R
