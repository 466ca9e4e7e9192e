"""A/B of the USE_FP16 render kernel (k_render_h) on the C4 scene; every variant must reproduce the first one's frame.
    python profiles/sweep_fp16.py [nx] [ny] [spp] [v1,v2,...] [n_spheres] [octree]
The USE_FP16 path has one kernel form (variant 0); an A/B partner gets a variant number of its own."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as entry

nx = int(sys.argv[1]) if len(sys.argv) > 1 else 960
ny = int(sys.argv[2]) if len(sys.argv) > 2 else 540
ns = int(sys.argv[3]) if len(sys.argv) > 3 else 4
variants = [int(x) for x in sys.argv[4].split(",")] if len(sys.argv) > 4 else [0]
n = int(sys.argv[5]) if len(sys.argv) > 5 else 100000
octree = int(sys.argv[6]) if len(sys.argv) > 6 else 1
spl = 300 if n > 10000 else 30
pkg = entry.load_package()
rt = pkg.RayTracer(0)
rt.create_world(n, 0.1, pkg.PREC_FP16)
if octree:
    print("build", rt.build_octree(spl, pkg.PREC_FP16))
rt.set_camera(nx, ny)
fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
ref = None
for v in variants:
    best = None
    for k in range(2):
        fb.zero_()
        st = rt.render_device(rt.args(nx, ny, ns, octree, precision=pkg.PREC_FP16, variant=v), fb.data_ptr())
        best = st if best is None or st["kernel_ms"] < best["kernel_ms"] else best
    if ref is None:
        ref = fb.clone()
    same = float((ref.view(torch.int32) == fb.view(torch.int32)).all(dim=2).float().mean())
    print(f"FP16 n={n} octree={octree} {nx}x{ny}x{ns} variant {v} kernel_ms {best['kernel_ms']:.3f} Mrays/s {best['rays'] / best['kernel_ms'] / 1e3:.1f} "
          f"identical_pixels {same} rays {best['rays']}", flush=True)
rt.close()
