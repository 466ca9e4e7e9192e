#!/usr/bin/env python
"""bench.py — the render hot path on N B200s, BASELINE.json's metric (Mrays/s, ms/frame).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C3|C1|C2|C5] [--shard tiles|spp] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (one rank per GPU, NCCL)

A "step" is one frame of the workload: render_init + render of the reference (main.cu:424-429), i.e. what its
"took X seconds" brackets.  `value` is whole-job Mrays/s (closest-hit queries / device time, max over ranks) with
the scene, octree and camera resident in HBM; `e2e` is the same metric through the public API with HOST buffers
(sphere descriptors uploaded, octree rebuilt, frame copied back to pinned host memory inside the timed region).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (n, spl, use_octree, nx, ny, ns, description)
    "C1": (488, 30, 0, 1200, 800, 10, "C1: RTIOW scene, 488 spheres, flat hitable_list, 1200x800, 10 spp, FP32"),
    "C2": (488, 30, 1, 1200, 800, 10, "C2: 488 spheres, octree SPHERES_PER_LEAF=30, 1200x800, 10 spp, FP32"),
    "C3": (100000, 300, 1, 3840, 2160, 64, "C3: 100k random spheres, octree SPHERES_PER_LEAF=300, 3840x2160, 64 spp, FP32"),
    "C4": (100000, 300, 1, 3840, 2160, 64, "C4: 100k random spheres, octree SPHERES_PER_LEAF=300, 3840x2160, 64 spp, USE_FP16"),
    "C5": (1000000, 3000, 1, 7680, 4320, 256, "C5: 1M random spheres, octree SPHERES_PER_LEAF=3000, 7680x4320, 256 spp, FP32"),
}
FP16_CONFIGS = {"C4"}
# CPU sample of the workload: every CPU_STRIDE-th pixel in x and y of the full frame, all ns samples
CPU_STRIDE = {"C1": (4, 4), "C2": (2, 2), "C3": (16, 16), "C4": (96, 96), "C5": (96, 96)}
# The reference's own CUDA build (oracle/_ref/ref_cuda_*: its kernels recompiled for sm_100).  `ref_cuda_leg` runs it LIVE on
# this box at REF_CUDA_LIVE_SPP samples (its create_world alone takes ~2 minutes at 100 k spheres: one thread device-news every
# material); the full 64-spp frame takes 3 minutes more, so that number is quoted from the committed record of
# tests/golden/gen_ref_cuda_full.sh (tests/golden/ref_cuda/manifest_full.json: render time per sample count, clocks under load).
REF_CUDA_BIN = {"C3": "ref_cuda_n100000_oct_spl300", "C4": "ref_cuda_n100000_oct_spl300_fp16"}
REF_CUDA_LIVE_SPP = 4
# --dump-outputs: frames up to this size are written whole, larger ones as a fixed, seeded sample of DUMP_SAMPLE_PIXELS pixels
DUMP_FULL_FRAME_BYTES = 48 << 20
DUMP_SAMPLE_PIXELS = 1 << 20
DUMP_SAMPLE_SEED = 1984


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def stop(self) -> dict:
        if self.proc:
            self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def cpu_reference_sample(cfg: str, threads: int = 0):
    """The reference's own code on the host cores (oracle/_ref/libref_host_*.so: its headers + color() compiled for
    the CPU, OpenMP over rows), or the oracle port when that library is absent.  Returns (Mrays/s, info)."""
    import __graft_entry__ as entry
    O = entry.load_oracle()
    n, spl, octree, nx, ny, ns, _ = CONFIGS[cfg]
    sx, sy = CPU_STRIDE[cfg]
    cores = threads or os.cpu_count() or 1
    params = O.make_params(nx, ny, ns, octree, spl, O.ARITH_HOST, step=(sx, sy), threads=cores)
    sample = f"pixels (i%{sx}==0, j%{sy}==0) of the {nx}x{ny} frame, all {ns} spp"
    variant = f"{'oct' if octree else 'brute'}_spl{spl}" + ("_fp16" if cfg in FP16_CONFIGS else "")
    if O.RefHost.available(variant):
        rh = O.RefHost(variant).create_world(n, 0.1, nx, ny)
        saved, devnull = os.dup(1), os.open(os.devnull, os.O_WRONLY)
        os.dup2(devnull, 1)            # the reference printf's when it drops spheres
        try:
            if octree:
                rh.build_octree()
            t0 = time.perf_counter()
            _, _, ctr = rh.render(params)
            dt = time.perf_counter() - t0
        finally:
            os.dup2(saved, 1)
            os.close(saved)
            os.close(devnull)
        rh.destroy()
        kind = "reference"
    else:
        sph, _ = O.create_world(n)
        blob = O.build_octree(sph, spl)[0] if octree else None
        cam = O.camera(nx, ny, O.ARITH_HOST)
        t0 = time.perf_counter()
        _, _, ctr = O.render(sph, cam, params, blob)
        dt = time.perf_counter() - t0
        kind = "port"
    return ctr["rays"] / dt / 1e6, {"cores": cores, "kind": kind, "sample": sample, "seconds": dt, "rays": ctr["rays"]}


def ref_cuda_leg(cfg: str, rays_at_live_spp: float, rays_full: float, budget_s: float):
    """Mrays/s of the reference's CUDA build on this box.  Live: REF_CUDA_LIVE_SPP samples per pixel of the same frame (clocks
    sampled while it runs).  Recorded: the committed timing of the full sample count.  Rays are counted by this repo's kernel
    for the same frame and sample count (identical sample chains, so identical ray counts)."""
    n, spl, octree, nx, ny, ns, _ = CONFIGS[cfg]
    out = {"binary": "oracle/_ref/" + REF_CUDA_BIN.get(cfg, "")}
    try:
        man = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_cuda", "manifest_full.json")))["timing"].get(cfg)
        if man:
            full = [r for r in man["runs"] if r["ns"] == ns]
            out["recorded"] = {"runs": man["runs"], "clocks": man["clocks"], "source": "tests/golden/ref_cuda/manifest_full.json"}
            if full and rays_full:
                out["recorded"]["ms_per_frame"] = full[0]["render_ms"]
                out["recorded"]["mrays_s"] = rays_full / full[0]["render_ms"] / 1e3
    except Exception as e:
        out["recorded"] = {"error": str(e)}
    exe = os.path.join(ROOT, "oracle", "_ref", REF_CUDA_BIN.get(cfg, "missing"))
    if not os.path.exists(exe):
        out["live"] = {"error": "binary not built (make -C oracle ref_cuda REF=<checkout of the reference>)"}
        return out
    if budget_s < 150:
        out["live"] = {"skipped": f"only {budget_s:.0f} s of the bench's time budget left; the run needs ~125 s (create_world alone ~115 s)"}
        return out
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    sampler.start()
    try:
        # (--reps 1 --no-free: the reference's free_world deletes 100 k materials from one device thread, another ~90 s)
        r = subprocess.run([exe, str(nx), str(ny), str(REF_CUDA_LIVE_SPP), "--reps", "1", "--no-free"], capture_output=True, text=True,
                           timeout=min(budget_s, 170))
        rec = json.loads(r.stdout.strip().splitlines()[-1])
        out["live"] = {"spp": REF_CUDA_LIVE_SPP, "render_ms": rec["render_ms"], "create_world_ms": rec["create_world_ms"],
                       "mrays_s": rays_at_live_spp / rec["render_ms"] / 1e3 if rays_at_live_spp else None,
                       "note": "render_init + render of the reference (main.cu:424-429), cudaEvent-timed; its per-sample cost grows with "
                               "the sample count (see recorded.runs), so the 64-spp ratio is larger than this one"}
    except Exception as e:
        out["live"] = {"error": str(e)[:200]}
    out["live_clocks"] = sampler.stop()
    return out


def run_reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path, all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cfg = args.config
    n, spl, octree, nx, ny, ns, desc = CONFIGS[cfg]
    vals, info = [], None
    for _ in range(max(0, args.warmup if args.warmup < 2 else 1)):      # CPU code needs no GPU-style warm-up
        pass
    t_all = time.perf_counter()
    for _ in range(args.steps):
        v, info = cpu_reference_sample(cfg)
        vals.append(v)
    value = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * (time.perf_counter() - t_all) / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": desc, "n_spheres": n, "spheres_per_leaf": spl, "use_octree": octree, "nx": nx, "ny": ny, "ns": ns},
            "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": info["cores"], "kind": info["kind"], "sample": info["sample"]},
            "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def dump_outputs(out_dir: str, fb, rays: float, paths: float):
    """What the timed path handed its caller in the last timed step: the finished frame (float32 [ny, nx, 3] on the device) and
    the ray and path counts.  A frame larger than DUMP_FULL_FRAME_BYTES is written as the same seeded pixel sample on every run
    (frame_sample.npy [K, 3] float32, frame_sample_pixels.npy [K] float64: linear index j * nx + i)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    ny, nx, _ = fb.shape
    if fb.numel() * 4 <= DUMP_FULL_FRAME_BYTES:
        np.save(os.path.join(out_dir, "frame.npy"), fb.cpu().numpy())
    else:
        rng = np.random.default_rng(DUMP_SAMPLE_SEED)
        pix = np.sort(rng.choice(nx * ny, size=min(DUMP_SAMPLE_PIXELS, nx * ny), replace=False))
        sample = fb.reshape(-1, 3)[torch.from_numpy(pix).to(fb.device)].cpu().numpy()
        np.save(os.path.join(out_dir, "frame_sample.npy"), sample)
        np.save(os.path.join(out_dir, "frame_sample_pixels.npy"), pix.astype(np.float64))
    np.save(os.path.join(out_dir, "ray_counts.npy"), np.array([rays, paths], dtype=np.float64))


def measure_e2e(pkg, mg, rt, torch, dist, dev, rank, world, mode, prec, n, spl, octree, nx, ny, ns, frame, fb, steps):
    """The same metric through the public API with HOST buffers, all N ranks taking part: host->device copy of the sphere
    descriptors, GPU octree build, (sharded) render, the reduce-scatter, /ns + sqrt of each rank's slice and its device->host copy
    into ONE pinned host frame (N = 1: rt_render_to_host; N > 1: a POSIX shared-memory frame every rank maps and page-locks, so the
    N slices cross PCIe in parallel).  Wall clock around barriers: max over ranks by construction."""
    import ctypes as C
    spheres = rt.spheres()
    host, host_fb = None, None
    if world == 1:
        host_fb = torch.empty((ny, nx, 3), dtype=torch.float32).pin_memory()
    else:
        name = f"rt_b200_frame_{os.environ.get('MASTER_PORT', '0')}_{os.getppid()}"
        if rank == 0:
            host = mg.SharedHostFrame(name, nx * ny * 12, True, torch)
        dist.barrier()
        if rank != 0:
            host = mg.SharedHostFrame(name, nx * ny * 12, False, torch)
        frame.attach_host(host)
    rays, secs = 0.0, 0.0
    phases = [0.0, 0.0, 0.0]           # rank 0's host clock: scene upload, octree build, render + exchange + copy-out
    for k in range(steps + 1):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rt.upload_world(spheres)
        ta = time.perf_counter()
        if octree:
            rt.build_octree(spl, prec)
        tb = time.perf_counter()
        if world == 1:
            a = rt.args(nx, ny, ns, octree, precision=prec)
            stt = pkg.RenderStats()
            rt._ck(rt.L.rt_render_to_host(rt._ctx, C.byref(a), C.c_void_p(host_fb.data_ptr()), C.byref(stt)), "rt_render_to_host")
            r = float(stt.rays)
        else:
            st = mg.render_sharded(rt, frame, ns, bool(octree), mode, dist, want_stats=True, to_host=True)
            r = float(st["rays"])
        torch.cuda.synchronize()
        tc = time.perf_counter()
        if world > 1:
            dist.barrier()
        dt = time.perf_counter() - t0
        if k > 0:
            phases[0] += ta - t0; phases[1] += tb - ta; phases[2] += tc - tb
        if world > 1:
            t = torch.tensor([r], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            r = float(t[0])
        if k > 0:                      # the first pass warms the allocations
            rays += r
            secs += dt
    check = None
    if world > 1:
        # what the N-GPU run left in the host frame, against the 1-GPU frame of the same config rendered on rank 0
        if rank == 0:
            got = host.array.reshape(ny, nx, 3).copy()
            one = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
            rt.render_device(rt.args(nx, ny, ns, octree, precision=prec), one.data_ptr())
            ref = one.cpu().numpy()
            import numpy as np
            fin = np.isfinite(got).all(axis=2) & np.isfinite(ref).all(axis=2)
            mse = float(((np.clip(got[fin], 0, 1) - np.clip(ref[fin], 0, 1)) ** 2).mean())
            check = {"sharding": "tiles" if mode == pkg.SHARD_TILES else "spp",
                     "identical_to_1gpu_frame": bool(np.array_equal(got.view(np.uint32), ref.view(np.uint32))),
                     "pixels_identical": float((got.view(np.uint32) == ref.view(np.uint32)).all(axis=2).mean()),
                     "mean_radiance": float(got[fin].mean()), "mean_radiance_1gpu": float(ref[fin].mean()),
                     "psnr_db_vs_1gpu": None if mse == 0 else float(10 * np.log10(1.0 / mse)),
                     "expect": "tiles: bit-identical; spp: same mean radiance, PSNR bounded by Monte-Carlo noise (independent streams)"}
        dist.barrier()
        frame.attach_host(None)
        host.close()
    return {"value": rays / secs / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(n * 36) * world,
            "d2h_bytes_per_step": int(nx * ny * 12 + 40), "ms_per_step": 1e3 * secs / steps, "frame_check": check,
            "phases_ms_rank0": {"scene_upload": 1e3 * phases[0] / steps, "octree_build": 1e3 * phases[1] / steps,
                                "render_exchange_copy": 1e3 * phases[2] / steps},
            "includes": "per rank: scene upload + GPU octree build + render of its shard; one reduce-scatter; /ns + sqrt and the copy of every "
                        "rank's slice into one pinned host frame"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS))
    ap.add_argument("--shard", default="spp", choices=["tiles", "spp"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip the live run of the reference's CUDA build (~130 s, N = 1 only)")
    ap.add_argument("--time-budget", type=float, default=330.0, help="seconds the whole bench may take; the reference-CUDA leg is skipped "
                                                                       "when less than 150 s of it are left")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU path computed: use it with --impl ours")
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    import __graft_entry__ as entry
    pkg = entry.load_package()
    from dd2360_raytracing_b200 import multigpu as mg

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    n, spl, octree, nx, ny, ns, desc = CONFIGS[args.config]
    prec = pkg.PREC_FP16 if args.config in FP16_CONFIGS else pkg.PREC_FP32
    if prec == pkg.PREC_FP16 and world > 1:
        raise SystemExit("the USE_FP16 config renders whole frames on one GPU (the half accumulator does not split); use --gpus 1")
    rt = pkg.RayTracer(local_rank)
    stream = torch.cuda.current_stream()
    rt.set_stream(stream.cuda_stream)
    rt.create_world(n, 0.1, prec)
    bst = rt.build_octree(spl, prec) if octree else None
    rt.set_camera(nx, ny)
    frame = mg.ShardedFrame(torch, dev, nx, ny, rank, world) if world > 1 else None
    fb = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev) if world == 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
    mode = pkg.SHARD_TILES if args.shard == "tiles" else pkg.SHARD_SPP

    def step(want_stats):
        if world == 1:
            return rt.render_device(rt.args(nx, ny, ns, octree, precision=prec), fb.data_ptr(), want_stats=want_stats)
        return mg.render_sharded(rt, frame, ns, bool(octree), mode, dist, want_stats=want_stats)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 0)):
        step(False)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    rays_local, kernel_ms, kernel_name = 0, [], None
    t_bench0 = time.perf_counter()
    barrier()
    for k in range(args.steps):
        flush.zero_()                                  # L2 flush between timed iterations (untimed)
        ev[k][0].record(stream)
        st = step(True)                                # reads the ray counter back: syncs the stream
        ev[k][1].record(stream)
        rays_local += st["rays"]
        kernel_ms.append(st["kernel_ms"])
        kernel_name = st["kernel"]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    t = torch.tensor([sum(step_ms), float(rays_local)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        total_ms, total_rays = float(tmax[0]), float(tsum[1])
    else:
        total_ms, total_rays = float(t[0]), float(t[1])
    if args.dump_outputs:
        last = torch.tensor([float(st["rays"]), float(st["paths"])], dtype=torch.float64, device=dev)
        out = fb
        if world > 1:                                  # every rank holds its finished slice of the flattened frame
            dist.all_reduce(last, op=dist.ReduceOp.SUM)
            whole = torch.empty(frame.S * world, dtype=torch.float32, device=dev)
            dist.all_gather_into_tensor(whole, frame.slice)
            out = whole[:frame.total].view(ny, nx, 3)
        if rank == 0:
            dump_outputs(args.dump_outputs, out, float(last[0]), float(last[1]))
    e2e_result = measure_e2e(pkg, mg, rt, torch, dist, dev, rank, world, mode, prec, n, spl, octree, nx, ny, ns, frame, fb, args.steps)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    value = total_rays / (total_ms * 1e-3) / 1e6
    launches_per_step = 1 if world == 1 else 2          # render + finalize of the rank's slice; the reduce-scatter is NCCL's kernel
    line = {"metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16" if prec == pkg.PREC_FP16 else "f32", "data": "synthetic",
            "config": {"workload": desc, "n_spheres": n, "spheres_per_leaf": spl, "use_octree": octree, "nx": nx, "ny": ny, "ns": ns,
                       "max_depth": 50, "seed": "curand_init(1984+pixel_index,0,0)", "sharding": "none" if world == 1 else args.shard,
                       "sharding_note": None if world == 1 else (
                           "spp: rank g traces ns/N samples of every pixel from its own XORWOW streams (g = 0: the reference's); a valid "
                           "frame of the same quality, not bit-identical to the 1-GPU frame.  --shard tiles is bit-identical (tests) but "
                           "keeps every pixel's whole sample chain on one GPU, so the longest chain bounds the frame time"),
                       "collective": None if world == 1 else "one NCCL reduce-scatter (sum) of the linear radiance buffer per frame; every rank "
                                                             "finalises its own slice",
                       "l2": "flushed between timed steps (256 MiB memset, untimed); each step times one whole frame",
                       "rays_per_frame": total_rays / args.steps, "octree_build_ms": bst["build_ms"] if bst else None},
            "clocks": clocks, "gpu_launches": launches_per_step * args.steps,
            "kernel_ms_per_step": sum(kernel_ms) / len(kernel_ms)}
    line["kernel"] = kernel_name

    # ---- end to end through the public API with HOST buffers: every rank uploads the sphere descriptors and rebuilds the
    #      octree, renders its shard, the shards are reduced, rank 0 copies the frame to pinned host memory ----
    line["e2e"] = e2e_result
    # ---- roofline of the dominant kernel (k_render): FP32 issue, SURVEY §8(d) formula with measured S, B ----
    try:
        if prec == pkg.PREC_FP16:
            # USE_FP16: the work is the exhaustive pair scan (DESIGN.md §5): 2 spheres per packed pair, 13 HFMA2-class instructions
            # per pair = 26 half flop per sphere in the filter; roots, node tests and shading are < 15 % of the instructions
            hpeak = rt.hfma2_peak_tflops()
            rti = pkg.RayTracer(local_rank, instrumented=True)
            rti.create_world(n, 0.1, prec)
            if octree:
                rti.build_octree(spl, prec)
            probe = torch.empty((ny // 8, nx // 8, 3), dtype=torch.float32, device=dev)
            ps = rti.render_device(rti.args(nx // 8, ny // 8, 1, octree, precision=prec), probe.data_ptr())
            rti.close()
            S = ps["sphere_tests"] / ps["rays"]
            flop_per_ray = 26.0 * S
            km = sum(kernel_ms) / len(kernel_ms)
            achieved = (total_rays / args.steps) * flop_per_ray / (km * 1e-3) / 1e12
            line["roofline"] = {"bound": "fp16 (packed HFMA2 issue)", "achieved": achieved, "peak": hpeak, "unit": "TFLOP/s", "frac": achieved / hpeak,
                                "traffic": None, "kernel": kernel_name, "flop_per_ray": flop_per_ray, "sphere_tests_per_ray": S,
                                "peak_source": "measured here: dense HFMA2 microbenchmark (rt_hfma2_peak), 4 flop per instruction",
                                "note": "the half-precision closest hit is an exhaustive scan of every sphere of every cell the ray's line crosses "
                                        "(the reference's candidate set; half arithmetic makes hits non-local and the test order part of the result), "
                                        "counted by the instrumented build on a 1/64 frame; HBM traffic is the frame"}
            raise StopIteration
        peak = rt.ffma_peak_tflops()
        rti = pkg.RayTracer(local_rank, instrumented=True)
        rti.create_world(n, 0.1)
        if octree:
            rti.build_octree(spl)
        probe = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
        ps = rti.render_device(rti.args(nx, ny, 1, octree), probe.data_ptr())
        S, B = ps["sphere_tests"] / ps["rays"], ps["node_tests"] / ps["rays"]
        flop_per_ray = 5 + 18 * S + 12 * B + 80
        km = sum(kernel_ms) / len(kernel_ms)
        achieved = (total_rays / args.steps / world) * flop_per_ray / (km * 1e-3) / 1e12
        traffic, inputs = None, {}
        pj = os.path.join(ROOT, "profiles", "roofline_inputs.json")
        if os.path.exists(pj):
            inputs = json.load(open(pj)).get(args.config, {})
            if not (kernel_name or "").startswith(inputs.get("kernel_prefix", "\0")):
                inputs = {}                      # the committed capture is of another kernel than the one that just ran
            traffic = inputs.get("dram_bytes_per_launch")
        line["roofline"] = {"bound": "fp32", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                            "traffic": traffic, "kernel": kernel_name, "flop_per_ray": flop_per_ray,
                            "sphere_tests_per_ray": S, "node_tests_per_ray": B,
                            "peak_source": "measured here: dense FFMA microbenchmark (rt_ffma_peak); MEASURED_PEAKS.json has no FP32 figure",
                            "note": "FP32 issue is the bounding unit (SURVEY §8d); HBM traffic is the 12 B/pixel frame only"}
        rti.close()
        # the unit that actually bounds it: warp-instruction issue slots (4 schedulers per SM, one warp instruction per
        # cycle each).  Instructions per ray come from the committed ncu capture of this kernel (profiles/), the rate is live.
        try:
            wpr = inputs.get("warp_instructions_per_ray")
            info = rt.device_info()
            if wpr:
                issue_peak = info["sm_count"] * 4 * info["clock_khz"] * 1e3
                issue_ach = (total_rays / args.steps / world) * wpr / (km * 1e-3)
                line["roofline_issue"] = {"bound": "issue", "achieved": issue_ach / 1e9, "peak": issue_peak / 1e9, "unit": "Gwarp-inst/s",
                                          "frac": issue_ach / issue_peak, "warp_instructions_per_ray": wpr,
                                          "active_lanes_per_instruction": inputs.get("active_lanes_per_instruction"),
                                          "source": inputs.get("warp_instructions_source"),
                                          "note": "instructions per ray from profiles/roofline_inputs.json (ncu smsp__inst_executed.sum), rate measured here"}
        except Exception:
            pass
        # the same kernel against the HBM roofline, for the record: algorithmic bytes = the 12 B/pixel frame
        hbm_peak = None
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
        except Exception:
            pass
        hbm_peak = hbm_peak or 6554.2
        hbm_achieved = (nx * ny * 12) / (km * 1e-3) / 1e9
        line["roofline_hbm"] = {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_achieved / hbm_peak,
                                "traffic": traffic, "note": "not the bounding unit: the path writes one frame and re-reads an L2-resident scene"}
    except StopIteration:
        pass
    except Exception as e:                                     # the roofline probe must never cost the bench line
        line["roofline"] = {"bound": "fp32", "error": str(e)}

    # ---- reported CPU baseline: the reference's own code on this box's host cores, bounded sample ----
    if world == 1 and not args.no_cpu_baseline:
        try:
            v, info = cpu_reference_sample(args.config)
            line["cpu_baseline"] = {"value": v, "unit": "Mrays/s", "cores": info["cores"], "kind": info["kind"],
                                    "sample": info["sample"], "seconds": info["seconds"]}
        except Exception as e:
            line["cpu_baseline"] = {"error": str(e)}
    # ---- the bar north_star sets: the reference's own CUDA build on this box ----
    if world == 1 and args.config in REF_CUDA_BIN and not args.no_ref_cuda:
        try:
            probe = torch.empty((ny, nx, 3), dtype=torch.float32, device=dev)
            r4 = rt.render_device(rt.args(nx, ny, REF_CUDA_LIVE_SPP, octree, precision=prec), probe.data_ptr())["rays"]
            del probe
            line["ref_cuda"] = ref_cuda_leg(args.config, float(r4), total_rays / args.steps, args.time_budget - (time.perf_counter() - t_bench0))
        except Exception as e:
            line["ref_cuda"] = {"error": str(e)[:200]}
    print(json.dumps(line), flush=True)
    rt.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
