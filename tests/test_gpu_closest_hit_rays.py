"""GPU tier (-m gpu): every FP32 closest-hit walk of the render kernels, through rt.trace_rays, ray by ray against the oracle on the ray
families of tests/ray_families.py, in three layouts each (as generated, shuffled, and 32k + r rays so that the cooperative hook's last
warp is partial).  The walk is chosen by RT_RENDER_VARIANT, which rt_create reads, so every walk gets a fresh RayTracer:
  octree    : 1 the per-lane trace_tree, 0 the default cooperative walk (coop_trace<2>; coop_trace<4> at 1 000 000 spheres);
  flat list : 20 the N-test sweep, 1 trace_tree over the grid of all spheres, 0 / 40 the cooperative walk over it (world_dense:
              four candidates per lane); every walk must also return the sweep's answer.
Which scenes get four candidates per lane is checked on the host build of the same grid (ray_families.Grid.long_lists).
Bar: sphere index and t bit-identical to the oracle (ties: tie_key), and in every family at least one hit on a sphere other than
the ground.  The input classes DESIGN §3
leaves outside the contract (ray_families.outside_contract) are left out and counted.  Rays per family: RAYS (3 000; 1 000 for flat
lists above 10 000 spheres and for the 1 000 000-sphere octree, whose oracle queries cost the most): about 1.1e5 traced rays per
scene and walk over the five layouts, 4e4 at 1 000 000 spheres; per-walk ray and hit counts are printed.  The file runs in 33 s on
one B200 (1 000 W power limit), most of it in the 1 000 000-sphere test's oracle queries on the host."""
import numpy as np
import pytest

import ray_families as F
import test_caller_worlds_host as W

pytestmark = pytest.mark.gpu

RAYS, RAYS_LARGE = 3000, 1000
SPL = 30


def _tracer(pkg, monkeypatch, variant, sph, octree, spl):
    monkeypatch.setenv("RT_RENDER_VARIANT", str(variant))
    rt = pkg.RayTracer(0)
    rt.upload_world(sph)
    if octree:
        rt.build_octree(spl)
    return rt


def _rays(hostsim, O, sph, blob, spl, octree, per_family, seed, long_lists=None):
    """{family: (org, dirs, oracle index, oracle t)} with the rays outside the contract left out.  long_lists: whether the grid's
    voxel lists must (True) or must not (False) send the cooperative walk to four candidates per lane (select_walk's rule)."""
    g = F.grid_geometry(hostsim, sph, blob, spl, octree)
    if long_lists is not None:
        assert g.long_lists() == long_lists, (g.voxels, g.refs)
    out = {}
    for fi, (family, make) in enumerate(F.FAMILIES.items()):
        org, dirs = make(sph, g, seed + fi, per_family)
        keep = ~F.outside_contract(org, dirs, octree)
        org, dirs = org[keep], dirs[keep]
        want_i, want_t = O.closest_hits(sph, org, dirs, blob, spl, octree)
        assert (want_i > 0).any(), f"family {family} hits no sphere but the ground"
        out[family] = (org, dirs, want_i, want_t)
    return out


def _check_walks(pkg, monkeypatch, sph, blob, spl, octree, rays, variants, subset=None):
    """Every variant, family and layout against the oracle; in flat-list mode also against variant 20's answer."""
    sweep = {}
    report = {}
    for v in variants:
        rt = _tracer(pkg, monkeypatch, v, sph, octree, spl)
        try:
            nrays = nhits = 0
            for fi, (family, (org, dirs, want_i, want_t)) in enumerate(rays.items()):
                if subset and v in subset:
                    org, dirs, want_i, want_t = (a[: len(a) // subset[v]] for a in (org, dirs, want_i, want_t))
                for lname, ix in F.layouts(len(org), fi):
                    got_i, got_t = rt.trace_rays(org[ix], dirs[ix], octree)
                    bad = F.first_mismatch(want_i[ix], want_t[ix], got_i, got_t)
                    assert bad is None, f"layout {lname}: {bad[1]} rays differ; " + F.describe(
                        family, f"RT_RENDER_VARIANT={v}", int(ix[bad[0]]), org, dirs, (int(want_i[ix][bad[0]]), float(want_t[ix][bad[0]])),
                        (int(got_i[bad[0]]), float(got_t[bad[0]])))
                    if not octree and lname == "generated":
                        if v == 20:
                            sweep[family] = (got_i, got_t)
                        elif family in sweep:
                            s_i, s_t = sweep[family]
                            assert F.first_mismatch(s_i[: len(got_i)], s_t[: len(got_i)], got_i, got_t) is None, (family, v)
                    nrays += len(ix)
                    nhits += int((got_i >= 0).sum())
            report[v] = (nrays, nhits)
        finally:
            rt.close()
    print(f"variant: (rays, hits) {report}")


@pytest.mark.parametrize("n,spl", [(488, 30), (8000, 30), (20000, 30), (100000, 300)])
def test_octree_walks_match_the_oracle_ray_by_ray(pkg, hostsim, O, monkeypatch, n, spl):
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    rays = _rays(hostsim, O, sph, blob, spl, True, RAYS, 7000 + n, long_lists=False)
    _check_walks(pkg, monkeypatch, sph, blob, spl, True, rays, (1, 0))


def test_one_million_sphere_octree_walks_match_the_oracle_ray_by_ray(pkg, hostsim, O, monkeypatch):
    """coop_trace<4> (the default at this size: voxel lists average 40 or more references) on every ray, trace_tree on a quarter."""
    sph, _ = O.create_world(1000000)
    blob, _ = O.build_octree(sph, 3000)
    rays = _rays(hostsim, O, sph, blob, 3000, True, RAYS_LARGE, 91, long_lists=True)
    _check_walks(pkg, monkeypatch, sph, blob, 3000, True, rays, (0, 1), subset={1: 4})


LIST_WORLDS = {
    "n488": lambda O: O.create_world(488)[0],
    "n6000": lambda O: O.create_world(6000)[0],
    "n20000": lambda O: O.create_world(20000)[0],
    "cloud60000": lambda O: W.world_cloud(60000, seed=22, half=8.0, height=16.0),
    "dense": lambda O: W.world_dense(),
}


@pytest.mark.parametrize("world", list(LIST_WORLDS))
def test_flat_list_walks_match_the_oracle_and_the_sweep(pkg, hostsim, O, monkeypatch, world):
    sph = LIST_WORLDS[world](O)
    per = RAYS if len(sph) <= 10000 else RAYS_LARGE
    rays = _rays(hostsim, O, sph, None, SPL, False, per, 5000 + len(sph), long_lists=world == "dense")
    _check_walks(pkg, monkeypatch, sph, None, SPL, False, rays, (20, 1, 0, 40))


@pytest.mark.parametrize("octree", [True, False], ids=["octree", "list"])
@pytest.mark.parametrize("world", ["hollow", "duplicates"])
def test_caller_world_walks_match_the_oracle(pkg, hostsim, O, monkeypatch, world, octree):
    """Hollow spheres (hit where |r| puts the surface) and exact duplicates (every hit a tie, ranked by tie_key / the index)."""
    sph = W.WORLDS[world]()
    blob = O.build_octree(sph, SPL)[0] if octree else None
    rays = _rays(hostsim, O, sph, blob, SPL, octree, RAYS, 3000 + len(world))
    _check_walks(pkg, monkeypatch, sph, blob, SPL, octree, rays, (1, 0) if octree else (20, 1, 0))
