"""Config 4 (USE_FP16: 100 k spheres, SPHERES_PER_LEAF 300, 3840x2160x64) in tile shards over N GPUs of one box.

    python profiles/fp16_shards.py OUT_DIR [--frames 3] [--ns 64]

bench.py renders C4 on one GPU only; this measures the USE_FP16 frame the way the RayTracing program shards it: one process,
one context per GPU, everything through the C ABI (RT_SHARD_TILES render, rt_reduce_scatter over NCCL, rt_finalize_ex(FP16)
on every rank's slice).  N = 1, then every N in {2, 4, 8} the box has; one warm-up frame and `--frames` timed frames each.
Per N: device ms (the slowest rank's kernel_ms, CUDA events), end-to-end ms (host clock around render, exchange,
rt_finalize_ex and a synchronise of every GPU), Mrays/s of both, and whether the frame is bit-identical to the 1-GPU frame.
Writes OUT_DIR/fp16_shards.json with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> list[dict]:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout
    return [dict(zip(("name", "power_limit"), (f.strip() for f in line.split(",")))) for line in out.strip().splitlines()]


def run(pkg, rts, N, nx, ny, ns, frames):
    import torch
    L = pkg.load_library()
    total = nx * ny * 3
    S = (total + N - 1) // N
    acc = [torch.zeros(S * N, dtype=torch.float32, device=f"cuda:{g}") for g in range(N)]
    sl = [torch.empty(S, dtype=torch.float32, device=f"cuda:{g}") for g in range(N)] if N > 1 else acc
    if N > 1:
        arr = (C.c_void_p * N)(*[r._ctx for r in rts[:N]])
        if L.rt_comm_init_all(arr, N) != 0:
            raise RuntimeError(L.rt_last_error(rts[0]._ctx).decode())
    shard = pkg.SHARD_TILES if N > 1 else pkg.SHARD_NONE
    args = [rts[g].args(nx, ny, ns, True, shard_mode=shard, shard_rank=g, shard_count=N, precision=pkg.PREC_FP16) for g in range(N)]

    def frame():
        for g in range(N):        # stats = NULL: the call returns once the kernel is queued, so the ranks render concurrently
            rts[g].render_accumulate(args[g], acc[g].data_ptr(), want_stats=False)
        if N > 1:
            assert L.rt_group_start() == 0
            for g in range(N):
                assert L.rt_reduce_scatter(rts[g]._ctx, C.c_void_p(acc[g].data_ptr()), C.c_void_p(sl[g].data_ptr()), S) == 0
            assert L.rt_group_end() == 0
        for g in range(N):
            rts[g].finalize_ex(sl[g].data_ptr(), sl[g].data_ptr(), S, ns, pkg.PREC_FP16)
        for g in range(N):
            rts[g].synchronize()

    for g in range(N):
        torch.cuda.synchronize(g)
    frame()                       # warm-up
    dev_ms, e2e_ms, rays = [], [], 0
    for _ in range(frames):
        t0 = time.perf_counter()
        frame()
        e2e_ms.append(1e3 * (time.perf_counter() - t0))
        st = [rts[g].last_render_stats() for g in range(N)]
        dev_ms.append(max(s["kernel_ms"] for s in st))
        rays = sum(s["rays"] for s in st)
    img = torch.cat([s.cpu() for s in sl])[:total].numpy().copy()
    if N > 1:
        for r in rts[:N]:
            L.rt_comm_destroy(r._ctx)
    dev, e2e = float(np.median(dev_ms)), float(np.median(e2e_ms))
    return img, {"gpus": N, "device_ms": dev, "device_ms_all": dev_ms, "e2e_ms": e2e, "e2e_ms_all": e2e_ms, "rays_per_frame": rays,
                 "mrays_per_s_device": rays / dev / 1e3, "mrays_per_s_e2e": rays / e2e / 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--ns", type=int, default=64)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    pkg = entry.load_package()
    nx, ny, n, spl = 3840, 2160, 100000, 300
    have = torch.cuda.device_count()
    counts = [1] + [k for k in (2, 4, 8) if k <= have]
    rts = [pkg.RayTracer(g) for g in range(max(counts))]
    for r in rts:
        r.create_world(n, 0.1, pkg.PREC_FP16)
        r.build_octree(spl, pkg.PREC_FP16)
        r.set_camera(nx, ny)
    rows, ref = [], None
    for N in counts:
        img, row = run(pkg, rts, N, nx, ny, a.ns, a.frames)
        if ref is None:
            ref = img
        row["bit_identical_to_1gpu"] = bool(((img.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(img) & np.isnan(ref))).all())
        row["speedup_device"] = rows[0]["device_ms"] / row["device_ms"] if rows else 1.0
        row["speedup_e2e"] = rows[0]["e2e_ms"] / row["e2e_ms"] if rows else 1.0
        rows.append(row)
        print(json.dumps(row), flush=True)
    for r in rts:
        r.close()
    out = {"config": "C4: 100 000 spheres, octree SPL 300, USE_FP16, 3840x2160", "ns": a.ns, "frames_timed": a.frames,
           "process_model": "one process, one context per GPU, C ABI: RT_SHARD_TILES + rt_reduce_scatter + rt_finalize_ex(FP16)",
           "gpus_on_box": have, "gpu": gpu_info(), "not_measured": [k for k in (2, 4, 8) if k > have], "runs": rows}
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "fp16_shards.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
