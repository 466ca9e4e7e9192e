"""Config 3 (100 k spheres, SPHERES_PER_LEAF 300, 3840x2160x64): the 1/16 x 1/16 pixel subsample through rt_render_pixels against
the full frame through rt_render, alternately in one process.

    python profiles/render_pixels_c3.py OUT_DIR [--rounds 3]

One warm-up call of each, then `--rounds` rounds of (frame, list); kernel_ms is the render's CUDA-event time (upstream seeding
off, so one launch each).  The list's values must equal the frame's at those pixels bit for bit.  Writes
OUT_DIR/render_pixels_c3.json with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from fp16_shards import gpu_info
    pkg = entry.load_package()
    nx, ny, ns, n, spl = 3840, 2160, 64, 100000, 300
    rt = pkg.RayTracer(0)
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).astype(np.uint32).reshape(-1)
    pix = torch.from_numpy(sub.view(np.int32)).cuda()
    out = torch.empty((len(sub), 3), dtype=torch.float32, device="cuda")
    fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    args = rt.args(nx, ny, ns, True)
    rt.render_device(args, fb.data_ptr())
    rt.render_pixels_device(args, pix.data_ptr(), len(sub), out.data_ptr())
    ms = {"frame": [], "list": []}
    st = {}
    for _ in range(a.rounds):
        st["frame"] = rt.render_device(args, fb.data_ptr())
        ms["frame"].append(st["frame"]["kernel_ms"])
        st["list"] = rt.render_pixels_device(args, pix.data_ptr(), len(sub), out.data_ptr())
        ms["list"].append(st["list"]["kernel_ms"])
    frame = fb.cpu().numpy().reshape(-1, 3)
    same = bool(np.array_equal(out.cpu().numpy().view(np.uint32), frame[sub].view(np.uint32)))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    res = {"config": "C3 3840x2160x64, 100 k spheres, SPHERES_PER_LEAF 300, one GPU", "pixels": {"frame": nx * ny, "list": len(sub)},
           "kernel_ms": ms, "median_ms": med, "speedup_frame_over_list": med["frame"] / med["list"],
           "rays": {k: int(v["rays"]) for k, v in st.items()}, "kernel": {k: v["kernel"] for k, v in st.items()},
           "list_equals_frame": same, "gpu": gpu_info()}
    print(json.dumps(res))
    rt.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "render_pixels_c3.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
