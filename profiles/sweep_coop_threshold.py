"""k_render (variant 1) against k_render_coop (variant 40) over the sphere count.
    python profiles/sweep_coop_threshold.py [nx ny spp]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as entry

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 3840
ny = int(sys.argv[2]) if len(sys.argv) > 2 else 2160
ns = int(sys.argv[3]) if len(sys.argv) > 3 else 8
pkg = entry.load_package()
rt = pkg.RayTracer(0)
fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
for n in (488, 2000, 8000, 20000, 50000, 100000, 300000, 1000000):
    spl = 30 if n <= 10000 else (300 if n <= 100000 else 3000)
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    rt.set_camera(nx, ny)
    out = []
    for v in (1, 40):
        best = min(rt.render_device(rt.args(nx, ny, ns if n < 1000000 else 2, True, variant=v), fb.data_ptr())["kernel_ms"] for _ in range(2))
        out.append(best)
    print(f"n={n}: k_render {out[0]:.2f} ms, k_render_coop {out[1]:.2f} ms; coop/lane speed {out[0] / out[1]:.2f}x", flush=True)
rt.close()
