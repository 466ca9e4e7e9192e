"""Run the render kernel a few times on one config — the command profiled with ncu (see profiles/README.md).
    python profiles/profile_render.py [C3] [spp] [launches]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as entry
from bench import CONFIGS

cfg = sys.argv[1] if len(sys.argv) > 1 else "C3"
n, spl, octree, nx, ny, ns, desc = CONFIGS[cfg]
ns = int(sys.argv[2]) if len(sys.argv) > 2 else ns
launches = int(sys.argv[3]) if len(sys.argv) > 3 else 3
variant = int(os.environ.get("RT_VARIANT", "0"))
pkg = entry.load_package()
rt = pkg.RayTracer(0)
rt.create_world(n, 0.1)
if octree:
    print("build", rt.build_octree(spl))
fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
for k in range(launches):
    st = rt.render_device(rt.args(nx, ny, ns, octree, variant=variant), fb.data_ptr())
    print(cfg, "spp", ns, "launch", k, "kernel_ms", round(st["kernel_ms"], 3), "Mrays/s", round(st["rays"] / st["kernel_ms"] / 1e3, 1))
rt.close()
if len(sys.argv) > 4 and sys.argv[4] == "counters":
    rti = pkg.RayTracer(0, instrumented=True)
    rti.create_world(n, 0.1)
    if octree:
        rti.build_octree(spl)
    st = rti.render_device(rti.args(nx, ny, 1, octree, variant=variant), fb.data_ptr())
    print("counters (1 spp): sphere_tests/ray", round(st["sphere_tests"] / st["rays"], 2), "visibility line tests/ray",
          round(st["node_tests"] / st["rays"], 3), "rays/path", round(st["rays"] / st["paths"], 3))
    rti.close()
