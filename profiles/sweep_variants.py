"""A/B: kernel variants of the octree render on one config; every variant must reproduce variant 0's frame bit for bit.
    python profiles/sweep_variants.py [C3] [spp] [v1,v2,...]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import __graft_entry__ as entry
from bench import CONFIGS

cfg = sys.argv[1] if len(sys.argv) > 1 else "C3"
n, spl, octree, nx, ny, ns, desc = CONFIGS[cfg]
ns = int(sys.argv[2]) if len(sys.argv) > 2 else 8
variants = [int(x) for x in sys.argv[3].split(",")] if len(sys.argv) > 3 else [0, 1, 31, 40]
pkg = entry.load_package()
rt = pkg.RayTracer(0)
rt.create_world(n, 0.1)
print("build", rt.build_octree(spl))
fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
ref = None
for v in variants:
    best = None
    for k in range(3):
        fb.zero_()
        try:
            st = rt.render_device(rt.args(nx, ny, ns, octree, variant=v), fb.data_ptr())
        except Exception as ex:
            print("variant", v, "FAILED:", ex, flush=True)
            break
        best = st if best is None or st["kernel_ms"] < best["kernel_ms"] else best
    if best is None:
        continue
    if ref is None:
        ref = fb.clone()
        ref_rays = best["rays"]
    same = float((ref == fb).all(dim=2).float().mean())
    print(cfg, "spp", ns, "variant", v, "kernel_ms", round(best["kernel_ms"], 3), "Mrays/s", round(best["rays"] / best["kernel_ms"] / 1e3, 1),
          "identical_pixels", same, "rays", best["rays"], "(ref", ref_rays, ")", flush=True)
rt.close()
