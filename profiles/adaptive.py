"""Adaptive sampling (rt_render_adaptive) against uniform frames at config 3 (100 k spheres, SPHERES_PER_LEAF 300, 3840x2160).

    python profiles/adaptive.py OUT_DIR [--ref-spp 1024]

The reference image is the uniform --ref-spp frame.  Runs: uniform 16, 32, 64 and 128 spp (rt_render), and adaptive with min_spp 8,
max_spp 256 and thresholds {0.5, 1, 2, 4}/255, and {8, 16, 32}/255 (at C3 the four small thresholds refine two thirds of the
frame to the budget).  For each run: device ms (stats.kernel_ms: the render kernel for uniform frames, the
whole call for adaptive ones), paths, mean spp, and MSE and PSNR (10 log10(1 / MSE), on the finalised float frame) against the
reference.  Every run is warmed up once (the adaptive one also grows its scratch).  Per adaptive round:
  * listed pixels, ms and Mrays/s: the round replayed through the public calls on the same buffers (two whole-frame progressive
    calls of min_spp/2, then for round r an rt_render_pixels_progressive call over window_pixels restricted to the tiles whose
    final count is above the round's count), so each round's ms is stats.kernel_ms of its list call (dedupe pass included);
  * selection-pass µs and the dedupe (preparation) kernel's µs inside the list call: from torch.profiler over one more adaptive
    call, in a run of its own.
Headline: the cheapest adaptive run whose PSNR reaches uniform-64's, against uniform-64's ms.  Writes OUT_DIR/adaptive_b200.json
with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

MIN_SPP, MAX_SPP = 8, 256
THRESHOLDS_255 = [0.5, 1.0, 2.0, 4.0, 8.0, 16.0, 32.0]
UNIFORM = [16, 32, 64, 128]


def quality(fb, ref):
    mse = float(np.mean((fb.astype(np.float64) - ref.astype(np.float64)) ** 2))
    return {"mse": mse, "psnr_db": 10.0 * math.log10(1.0 / mse)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--ref-spp", type=int, default=1024)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from fp16_shards import gpu_info
    pkg = entry.load_package()
    nx, ny, n, spl = 3840, 2160, 100000, 300
    npix = nx * ny
    rt = pkg.RayTracer(0)
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    fb = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
    accum = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
    state = torch.empty(npix * 6, dtype=torch.int32, device="cuda")
    counts = torch.empty(npix, dtype=torch.int32, device="cuda")
    err = torch.empty(npix, dtype=torch.float32, device="cuda")

    ref_st = rt.render_device(rt.args(nx, ny, a.ref_spp, True), fb.data_ptr())
    ref = fb.cpu().numpy().reshape(ny, nx, 3)

    uniform = {}
    for ns in UNIFORM:
        rt.render_device(rt.args(nx, ny, ns, True), fb.data_ptr())                  # warm-up
        st = rt.render_device(rt.args(nx, ny, ns, True), fb.data_ptr())
        uniform[ns] = {"ms": st["kernel_ms"], "paths": int(st["paths"]), "rays": int(st["rays"]), "spp": ns,
                       **quality(fb.cpu().numpy().reshape(ny, nx, 3), ref)}

    def adaptive(thr):
        return rt.render_adaptive_device(rt.args(nx, ny, MAX_SPP, True), MIN_SPP, thr, accum.data_ptr(), state.data_ptr(), counts.data_ptr(),
                                         fb.data_ptr(), err.data_ptr())

    from torch.profiler import ProfilerActivity, profile
    tiles = pkg.window_pixels(nx, ny, 0, nx, 0, ny)
    runs = {}
    for t255 in THRESHOLDS_255:
        thr = t255 / 255.0
        adaptive(thr)                                                                # warm-up
        st = adaptive(thr)
        cnt = counts.cpu().numpy().view(np.uint32)
        run = {"threshold": thr, "threshold_255": t255, "ms": st["kernel_ms"], "paths": int(st["paths"]), "rays": int(st["rays"]),
               "mean_spp": st["paths"] / npix, "rounds": st["rounds"], "round_pixels": st["round_pixels"],
               "spp_histogram": {int(k): int(v) for k, v in zip(*np.unique(cnt, return_counts=True))},
               **quality(fb.cpu().numpy().reshape(ny, nx, 3), ref)}
        # the rounds replayed through the public calls
        args = rt.args(nx, ny, MIN_SPP // 2, True)
        rt.render_progressive(args, accum.data_ptr(), state.data_ptr(), True)
        rt.render_progressive(args, accum.data_ptr(), state.data_ptr(), False)
        c, per_round = MIN_SPP, []
        while c < MAX_SPP and (cnt > c).any():
            more = min(c, MAX_SPP - c)
            lst = tiles[cnt[tiles] > c]           # round r's list: the tiles that went on past count c, in tile order
            d = torch.from_numpy(lst.view(np.int32)).cuda()
            s = rt.render_pixels_progressive(rt.args(nx, ny, more, True), d.data_ptr(), d.numel(), accum.data_ptr(), state.data_ptr())
            per_round.append({"pixels": len(lst), "ns": more, "ms": s["kernel_ms"], "rays": int(s["rays"]),
                              "mrays_per_s": s["rays"] / s["kernel_ms"] / 1e3})
            c += more
        assert [r["pixels"] for r in per_round] == st["round_pixels"], (per_round, st["round_pixels"])
        # selection passes and the dedupe pass, from the profiler's trace of one more call
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            adaptive(thr)
            torch.cuda.synchronize()
        sel, prep, k = [], [], -1
        for e in sorted((e for e in prof.events() if e.device_type.name == "CUDA"), key=lambda e: e.time_range.start):
            us = e.device_time if hasattr(e, "device_time") else e.cuda_time
            if "k_adaptive_select" in e.name:
                k += 1
                sel.append(0.0)
            if k >= 0 and ("k_adaptive_" in e.name or "DeviceScan" in e.name):
                sel[k] += us
            elif "k_pixels_progressive_prep" in e.name:
                prep.append(us)
        for r, pr in enumerate(per_round):
            pr["selection_us"] = sel[r] if r < len(sel) else None
            pr["dedupe_us"] = prep[r] if r < len(prep) else None
        run["per_round"] = per_round
        run["final_selection_us"] = sel[len(per_round)] if len(sel) > len(per_round) else None
        run["selection_us_total"] = float(sum(sel))
        runs[str(t255)] = run
        print(json.dumps({k: v for k, v in run.items() if k != "spp_histogram"}))

    u64 = uniform[64]
    reach = [r for r in runs.values() if r["psnr_db"] >= u64["psnr_db"]]
    best = min(reach, key=lambda r: r["ms"]) if reach else None
    headline = {"uniform64_ms": u64["ms"], "uniform64_psnr_db": u64["psnr_db"],
                "adaptive_reaching_uniform64": None if best is None else
                {"threshold_255": best["threshold_255"], "ms": best["ms"], "psnr_db": best["psnr_db"], "mean_spp": best["mean_spp"],
                 "speedup": u64["ms"] / best["ms"]}}
    res = {"config": f"C3 scene (100 k spheres, SPHERES_PER_LEAF 300), {nx}x{ny}, octree, one GPU, HEAD seeding; adaptive min_spp "
                     f"{MIN_SPP}, max_spp {MAX_SPP}",
           "reference": {"spp": a.ref_spp, "ms": ref_st["kernel_ms"]},
           "uniform": {str(k): v for k, v in uniform.items()}, "adaptive": runs, "headline": headline,
           "kernel": ref_st["kernel"], "gpu": gpu_info()}
    print(json.dumps(headline))
    rt.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "adaptive_b200.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
