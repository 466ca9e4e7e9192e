"""From how many spheres do flat voxels and the cooperative kernel pay?  k_render (variant 1) and k_render_coop (variant 40) on
cubic and flat voxels over the sphere count.
    python profiles/sweep_flat_threshold.py [nx ny spp]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as entry

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 3840
ny = int(sys.argv[2]) if len(sys.argv) > 2 else 2160
ns = int(sys.argv[3]) if len(sys.argv) > 3 else 8
pkg = entry.load_package()
fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
for n in (2000, 5000, 10000, 20000, 30000, 50000, 100000):
    spl = 30 if n <= 10000 else 300
    out = {}
    for shape in ("1:1:1", "1.5:0.75:1"):
        os.environ["RT_GRID_SHAPE"] = shape
        rt = pkg.RayTracer(0)
        rt.create_world(n, 0.1)
        rt.build_octree(spl)
        rt.set_camera(nx, ny)
        for v in (1, 40):
            out[(shape, v)] = min(rt.render_device(rt.args(nx, ny, ns, True, variant=v), fb.data_ptr())["kernel_ms"] for _ in range(3))
        rt.close()
    print(f"n={n}: k_render cubic {out[('1:1:1', 1)]:.2f} flat {out[('1.5:0.75:1', 1)]:.2f} ms; k_render_coop cubic {out[('1:1:1', 40)]:.2f} "
          f"flat {out[('1.5:0.75:1', 40)]:.2f} ms", flush=True)
