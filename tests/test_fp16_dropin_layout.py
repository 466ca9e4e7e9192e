"""CPU tier: the USE_FP16 Octree layout of include/rt_dropin.h (AABB of six halves, 48-byte nodes) and of
rt_octree_reference_bytes_ex, and the header's half -> float conversion.  No GPU needed."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r"""
#include <cstdio>
#include "rt_dropin.h"
int main(int argc, char **) {
    printf("%zu %zu %zu\n", sizeof(Octree), sizeof(OctNode), sizeof(AABB));
#ifdef USE_FP16
    if (argc > 1)                                   /* every half bit pattern through rt_half_storage's float conversion */
        for (unsigned b = 0; b < 65536u; b++) { rt_half_storage h{(uint16_t)b}; const float f = h; unsigned u; memcpy(&u, &f, 4); printf("%08x\n", u); }
#endif
    return 0;
}
"""


def _probe(tmp_path, pkg, defines, *args):
    src = tmp_path / "probe.cpp"
    src.write_text(PROBE)
    exe = str(tmp_path / ("probe" + "".join(d.replace("=", "_") for d in defines)))
    lib_dir = os.path.dirname(pkg.LIB_PATH)
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Werror", *defines, "-I", os.path.join(ROOT, "include"), str(src), "-o", exe,
                    f"-L{lib_dir}", "-lrt_b200", f"-Wl,-rpath,{lib_dir}"], check=True)
    return subprocess.run([exe, *args], capture_output=True, text=True, check=True).stdout.split()


@pytest.mark.parametrize("spl,fp16_bytes,fp32_bytes", [(30, 536116, 543136), (300, 4960876, 4967896), (3000, 49208476, 49215496)])
def test_octree_size_with_and_without_use_fp16(pkg, tmp_path, spl, fp16_bytes, fp32_bytes):
    """sizeof(Octree) of the reference's FP16 build (48-byte OctNode) and FP32 build (60-byte OctNode), from the drop-in header
    and from the library, which sizes the exported blob with it."""
    L = pkg.load_library()
    d = [f"-DSPHERES_PER_LEAF={spl}"]
    assert _probe(tmp_path, pkg, d) == [str(fp32_bytes), "60", "24"]
    assert _probe(tmp_path, pkg, d + ["-DUSE_FP16"]) == [str(fp16_bytes), "48", "12"]
    assert L.rt_octree_reference_bytes_ex(spl, pkg.PREC_FP16) == fp16_bytes
    assert L.rt_octree_reference_bytes_ex(spl, pkg.PREC_FP32) == fp32_bytes == L.rt_octree_reference_bytes(spl)


def test_octree_size_rejects_unknown_arguments(pkg):
    L = pkg.load_library()
    assert L.rt_octree_reference_bytes_ex(30, 7) == 0
    assert L.rt_octree_reference_bytes_ex(0, pkg.PREC_FP16) == 0


def test_half_storage_reads_every_half_as_numpy_does(pkg, tmp_path):
    out = _probe(tmp_path, pkg, ["-DUSE_FP16"], "all")
    got = np.array([int(x, 16) for x in out[3:]], dtype=np.uint32)
    want = np.arange(65536, dtype=np.uint32).astype(np.uint16).view(np.float16).astype(np.float32).view(np.uint32)
    nan = np.isnan(want.view(np.float32))
    assert np.array_equal(got[~nan], want[~nan])
    assert np.isnan(got[nan].view(np.float32)).all()
