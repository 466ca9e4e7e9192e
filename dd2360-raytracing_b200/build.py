"""Build driver for librt_b200.so (nvcc, sm_100a only).  Used by __graft_entry__.build() and the tests.

    python dd2360-raytracing_b200/build.py [--force] [--counters]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "librt_b200.so")
LIB_COUNTERS = os.path.join(HERE, "librt_b200_counters.so")   # same code with -DRT_COUNTERS: work counters for the roofline
CLI = os.path.join(HERE, "RayTracing")
SOURCES = ["rt_abi.cu", "rt_render.cu", "rt_octree.cu", "rt_ppm.cu", "rt_adaptive.cu"]
HEADERS = ["rt_math.cuh", "rt_types.h", "rt_shade.cuh", "rt_trace.cuh", "rt_coop.cuh", "rt_chain.cuh", "rt_xorwow_skip.h", "rt_half.cuh", "rt_render_half.cuh", "rt_build.cuh", "rt_octree.h", "rt_render.h", "rt_adaptive.h", "rt_buffer.h",
           os.path.join("..", "..", "include", "rt_abi.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--extended-lambda",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-Wno-deprecated-gpu-targets"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: librt_b200.so cannot be built (there is no CPU fallback)")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _build_lib(target: str, extra: list[str], tag: str, env: dict, verbose: bool) -> None:
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", f"{tag}.o"))
        objs.append(obj)
        cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-Xptxas", "-v", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {src}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    with open(os.path.join(HERE, "build", f"ptxas{tag}.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    subprocess.run([_nvcc(), "-shared", "-o", target, *objs, "-lcudart_static", "-lpthread", "-ldl", "-lrt"],
                   check=True, env=env)


def build(force: bool = False, verbose: bool = False) -> str:
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
    if force or _stale(LIB, deps):
        _build_lib(LIB, [], "", env, verbose)
    if force or _stale(LIB_COUNTERS, deps):
        _build_lib(LIB_COUNTERS, ["-DRT_COUNTERS"], "_counters", env, False)
    cli_src = os.path.join(CSRC, "raytracing_main.cpp")
    if os.path.exists(cli_src) and (force or _stale(CLI, [cli_src, LIB])):
        subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(HERE, "..", "include"), cli_src, "-o", CLI,
                        f"-L{HERE}", "-lrt_b200", "-lpthread", f"-Wl,-rpath,$ORIGIN"], check=True, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
