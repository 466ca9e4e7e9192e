"""One bench.py configuration on one GPU with two builds of librt_b200.so, alternately in one process.

    python profiles/ab_libs.py OTHER_LIB OUT_DIR [--config C4] [--rounds 3]

OTHER_LIB is another build of the library (e.g. the parent commit's); the other side is this tree's build.  Each round renders
one frame with each library (one warm-up frame each first) and records the render's kernel_ms (CUDA events); the frames of the
two builds must be bit-identical.  Writes OUT_DIR/ab_libs_<config>.json with the GPU's name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench import CONFIGS, FP16_CONFIGS  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other_lib")
    ap.add_argument("out_dir")
    ap.add_argument("--config", default="C4", choices=sorted(CONFIGS))
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from fp16_shards import gpu_info
    pkg = entry.load_package()
    n, spl, octree, nx, ny, ns, desc = CONFIGS[a.config]
    prec = pkg.PREC_FP16 if a.config in FP16_CONFIGS else pkg.PREC_FP32
    this = pkg.load_library()
    other = C.CDLL(os.path.abspath(a.other_lib))          # an older build may lack later entry points: bind what it exports
    for name in pkg.ABI_SYMBOLS:
        if hasattr(other, name):
            fn, ref = getattr(other, name), getattr(this, name)
            fn.restype, fn.argtypes = ref.restype, ref.argtypes
    libs = {"this_tree": this, "other": other}
    rts, fbs = {}, {}
    for name, lib in libs.items():
        pkg._lib = lib                    # RayTracer binds the library load_library() returns
        r = pkg.RayTracer(0)
        r.create_world(n, 0.1, prec)
        if octree:
            r.build_octree(spl, prec)
        rts[name], fbs[name] = r, torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        r.render_device(r.args(nx, ny, ns, octree, precision=prec), fbs[name].data_ptr())     # warm-up
    pkg._lib = libs["this_tree"]
    ms = {k: [] for k in rts}
    for _ in range(a.rounds):
        for name, r in rts.items():
            ms[name].append(r.render_device(r.args(nx, ny, ns, octree, precision=prec), fbs[name].data_ptr())["kernel_ms"])
    x, y = fbs["this_tree"].cpu().numpy(), fbs["other"].cpu().numpy()
    same = bool(((x.view(np.uint32) == y.view(np.uint32)) | (np.isnan(x) & np.isnan(y))).all())
    out = {"config": desc + ", one GPU", "other_lib": a.other_lib,
           "kernel_ms": ms, "median_ms": {k: float(np.median(v)) for k, v in ms.items()}, "frames_bit_identical": same, "gpu": gpu_info()}
    print(json.dumps(out))
    for r in rts.values():
        r.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, f"ab_libs_{a.config.lower()}.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
