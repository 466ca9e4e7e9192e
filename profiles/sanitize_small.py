"""A few small renders through every kernel shape, for compute-sanitizer (memcheck / racecheck / initcheck).
    compute-sanitizer --tool racecheck python profiles/sanitize_small.py"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as entry
pkg = entry.load_package()
rt = pkg.RayTracer(0)
for n, spl, nx, ny, ns, variants in ((8000, 30, 64, 40, 2, (0, 40, 1)), (100000, 300, 48, 27, 1, (0, 1))):
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    ref = None
    for v in variants:
        fb, st = rt.render(nx, ny, ns, use_octree=True, variant=v)
        if ref is None:
            ref = fb
        print(n, "variant", v, st["kernel"], "rays", st["rays"], "same", bool((fb.view("uint32") == ref.view("uint32")).all()), flush=True)
rt.close()
