"""Progressive pixel lists at config 3 (100 k spheres, SPHERES_PER_LEAF 300, 3840x2160): 4 more samples per call for the whole
frame (rt_render_progressive) and for pixel lists (rt_render_pixels_progressive) on the same frame-indexed buffers.

    python profiles/pixel_progressive.py OUT_DIR [--rounds 5]

Variants: the frame call; the whole frame as a list in 8x4 tile order (window_pixels); 10 % and 1 % of the pixels as centred
window_pixels rectangles and as uniformly random pixels in raster order (what np.nonzero of a per-pixel mask gives).  Every
variant is warmed up once, then `--rounds` rounds run them all in alternation; ms is the call's CUDA-event time (stats.kernel_ms:
the preparation pass and the render), Mrays/s = rays / ms.  The preparation pass on its own (bitmask clear + dedupe, counts and
seeding kernel) is timed with torch.profiler over one more call of each list, in a run of its own.  Writes
OUT_DIR/pixel_progressive.json with the GPU's name and power limit read in the same run.
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
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from fp16_shards import gpu_info
    pkg = entry.load_package()
    nx, ny, ns, n, spl = 3840, 2160, 4, 100000, 300
    npix = nx * ny
    rt = pkg.RayTracer(0)
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    rng = np.random.default_rng(2024)

    def window(frac):
        w, h = int(round(nx * frac ** 0.5)), int(round(ny * frac ** 0.5))
        i0, j0 = (nx - w) // 2, (ny - h) // 2
        return pkg.window_pixels(nx, ny, i0, i0 + w, j0, j0 + h)

    lists = {
        "list_whole_frame_tiles": pkg.window_pixels(nx, ny, 0, nx, 0, ny),
        "window_10pct": window(0.10),
        "window_1pct": window(0.01),
        "scattered_10pct": np.sort(rng.choice(npix, npix // 10, replace=False)).astype(np.uint32),
        "scattered_1pct": np.sort(rng.choice(npix, npix // 100, replace=False)).astype(np.uint32),
    }
    dev = {k: torch.from_numpy(v.view(np.int32)).cuda() for k, v in lists.items()}
    accum = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
    state = torch.empty(npix * 6, dtype=torch.int32, device="cuda")
    counts = torch.full((npix,), ns, dtype=torch.int32, device="cuda")
    args = rt.args(nx, ny, ns, True)
    rt.render_progressive(args, accum.data_ptr(), state.data_ptr(), True)

    def call(name):
        if name == "frame":
            st = rt.render_progressive(args, accum.data_ptr(), state.data_ptr(), False)
            counts.add_(ns)
            return st
        p = dev[name]
        return rt.render_pixels_progressive(args, p.data_ptr(), p.numel(), accum.data_ptr(), state.data_ptr(), counts.data_ptr())

    names = ["frame", *lists]
    for k in names:                                     # warm-up
        call(k)
    ms = {k: [] for k in names}
    last = {}
    for _ in range(a.rounds):
        for k in names:
            last[k] = call(k)
            ms[k].append(last[k]["kernel_ms"])
    med = {k: float(np.median(v)) for k, v in ms.items()}
    rays = {k: int(v["rays"]) for k, v in last.items()}

    # the preparation pass alone: device time of its kernel and of the bitmask clear, from the profiler's trace
    from torch.profiler import ProfilerActivity, profile
    prep = {}
    for k in lists:
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(k)
            torch.cuda.synchronize()
        us = {"prep_kernel_us": 0.0, "mask_clear_us": 0.0}
        for e in prof.events():
            if e.device_type.name != "CUDA":
                continue
            t = e.device_time if hasattr(e, "device_time") else e.cuda_time
            if "k_pixels_progressive_prep" in e.name:
                us["prep_kernel_us"] += t
            elif "memset" in e.name.lower():
                us["mask_clear_us"] += t
        prep[k] = us

    res = {"config": f"C3 scene (100 k spheres, SPHERES_PER_LEAF 300), {nx}x{ny}, {ns} more spp per call, one GPU, HEAD seeding",
           "pixels": {"frame": npix, **{k: len(v) for k, v in lists.items()}},
           "kernel_ms": ms, "median_ms": med, "rays": rays,
           "mrays_per_s": {k: rays[k] / med[k] / 1e3 for k in names},
           "ms_over_frame": {k: med[k] / med["frame"] for k in names},
           "rays_over_frame": {k: rays[k] / rays["frame"] for k in names},
           "kernel": {k: v["kernel"] for k, v in last.items()},
           "launches": {k: int(v["launches"]) for k, v in last.items()},
           "preparation_pass": prep, "gpu": gpu_info()}
    print(json.dumps(res))
    rt.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "pixel_progressive.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
