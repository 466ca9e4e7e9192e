"""Config 4 (USE_FP16, 3840x2160x64) on one GPU with two builds of librt_b200.so, alternately in one process.

    python profiles/ab_libs_c4.py OTHER_LIB OUT_DIR [--rounds 3]

OTHER_LIB is another build of the library (e.g. the parent commit's); the other side is this tree's build.  Each round renders
one frame with each library (one warm-up frame each first) and records the render's kernel_ms (CUDA events); the frames of the
two builds must be bit-identical.  Writes OUT_DIR/ab_libs_c4.json with the GPU's name and power limit read in the same run.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other_lib")
    ap.add_argument("out_dir")
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    import torch
    import __graft_entry__ as entry
    from fp16_shards import gpu_info
    pkg = entry.load_package()
    nx, ny, ns, n, spl = 3840, 2160, 64, 100000, 300
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
        r.create_world(n, 0.1, pkg.PREC_FP16)
        r.build_octree(spl, pkg.PREC_FP16)
        rts[name], fbs[name] = r, torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        r.render_device(r.args(nx, ny, ns, True, precision=pkg.PREC_FP16), fbs[name].data_ptr())     # warm-up
    pkg._lib = libs["this_tree"]
    ms = {k: [] for k in rts}
    for _ in range(a.rounds):
        for name, r in rts.items():
            ms[name].append(r.render_device(r.args(nx, ny, ns, True, precision=pkg.PREC_FP16), fbs[name].data_ptr())["kernel_ms"])
    x, y = fbs["this_tree"].cpu().numpy(), fbs["other"].cpu().numpy()
    same = bool(((x.view(np.uint32) == y.view(np.uint32)) | (np.isnan(x) & np.isnan(y))).all())
    out = {"config": "C4: 100 000 spheres, octree SPL 300, USE_FP16, 3840x2160x64, one GPU", "other_lib": a.other_lib,
           "kernel_ms": ms, "median_ms": {k: float(np.median(v)) for k, v in ms.items()}, "frames_bit_identical": same, "gpu": gpu_info()}
    print(json.dumps(out))
    for r in rts.values():
        r.close()
    os.makedirs(a.out_dir, exist_ok=True)
    with open(os.path.join(a.out_dir, "ab_libs_c4.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
