"""Known answers for curand_init(seed, subsequence, 0) from cuRAND ITSELF: the toolkit's curand_kernel.h compiled for the host
(nvcc; the same shim as oracle/ref_host_driver.cu: cuRAND's QUALIFIERS made __host__ __device__).  Needs nvcc, no GPU.

    python tests/golden/gen_curand_kat.py

writes
  tests/golden/curand_subsequence_kat.json   state words d, v0..v4 for chosen (seed, subsequence) pairs ("cases") and for the
                                              40 pairs tests/test_oracle.py draws with numpy's default_rng(3) ("random_cases")
  tests/golden/curand_upstream_60x40.npy      uint32 [2400, 6]: curand_init(1984, pixel_index, 0) for every pixel of a 60x40
                                              frame, the per-pixel states of the upstream seeding (main.cu:90)
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
GOLDEN = os.path.join(ROOT, "tests", "golden")

SRC = r"""
#define QUALIFIERS static __forceinline__ __host__ __device__
#include <curand_kernel.h>
#include <cstdio>
int main() {
    unsigned long long seed, sub;
    while (std::scanf("%llu %llu", &seed, &sub) == 2) {
        curandState s;
        curand_init(seed, sub, 0, &s);
        std::printf("%u %u %u %u %u %u\n", s.d, s.v[0], s.v[1], s.v[2], s.v[3], s.v[4]);
    }
    return 0;
}
"""


def curand_states(pairs):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    with tempfile.TemporaryDirectory() as d:
        src, exe = os.path.join(d, "curand_states.cu"), os.path.join(d, "curand_states")
        open(src, "w").write(SRC)
        subprocess.run([nvcc, "-O2", "-w", "-Wno-deprecated-gpu-targets", src, "-o", exe], check=True)
        out = subprocess.run([exe], input="".join(f"{s} {q}\n" for s, q in pairs), capture_output=True, text=True, check=True).stdout
    return [[int(x) for x in line.split()] for line in out.splitlines()]


def random_pairs():
    rr = np.random.default_rng(3)
    pairs = []
    for _ in range(40):
        pairs.append((int(rr.integers(0, 2 ** 63)), int(rr.integers(0, 2 ** 40))))
    return pairs


if __name__ == "__main__":
    cases = [(1984, s) for s in (0, 1, 2, 3, 4, 5, 7, 8, 15, 16, 255, 256, 1199, 1200, 65535, 65536, 959999, 8294399, 33177599,
                                  33177600, 2 ** 31 - 1, 2 ** 32 + 5, 2 ** 39 + 12345)]
    cases += [(0, 1), (1, 1), (7, 123456789), (2 ** 32 + 1984, 42), (2 ** 40 + 17, 77), (2 ** 63 + 3, 1000003)]
    rnd = random_pairs()
    pixels = [(1984, p) for p in range(60 * 40)]
    states = curand_states(cases + rnd + pixels)
    a, b = len(cases), len(cases) + len(rnd)
    out = {"source": "cuRAND 10.3.10 (CUDA 12.9 curand_kernel.h) host-compiled; state words d, v0..v4 after curand_init(seed, subsequence, 0)",
           "cases": [{"seed": s, "subsequence": q, "state": st} for (s, q), st in zip(cases, states[:a])],
           "random_cases": [{"seed": s, "subsequence": q, "state": st} for (s, q), st in zip(rnd, states[a:b])]}
    json.dump(out, open(os.path.join(GOLDEN, "curand_subsequence_kat.json"), "w"), indent=1)
    np.save(os.path.join(GOLDEN, "curand_upstream_60x40.npy"), np.array(states[b:], dtype=np.uint32))
    print(len(cases), "cases,", len(rnd), "random cases,", len(pixels), "pixel states written", file=sys.stderr)
