"""CPU tier: the C-ABI library loads, exports every symbol include/rt_abi.h declares, and fails loudly without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    txt = open(os.path.join(ROOT, "include", "rt_abi.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(rt_[a-z0-9_]+)\s*\(", txt)))


def test_header_and_binding_agree(pkg):
    assert _declared_symbols() == sorted(pkg.ABI_SYMBOLS)


def test_library_exports_every_declared_symbol(pkg):
    L = pkg.load_library()
    for name in _declared_symbols():
        assert hasattr(L, name), f"librt_b200.so does not export {name}"
    assert L.rt_abi_version() == 1


def test_no_torch_types_in_the_abi():
    txt = open(os.path.join(ROOT, "include", "rt_abi.h")).read()
    code = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    for banned in ("torch", "std::", "class ", "template", "&)"):
        assert banned not in code, banned


def test_struct_layouts(pkg, O):
    assert C.sizeof(pkg.RenderArgs) == 64
    assert pkg.SPHERE_DTYPE.itemsize == 36 and pkg.SPHERE_DTYPE == O.SPHERE_DTYPE
    assert C.sizeof(pkg.CameraDesc) == 52


def test_reference_octree_size(pkg):
    # sizeof(Octree) for SPHERES_PER_LEAF = 30 / 300 / 3000 (SURVEY A.3)
    L = pkg.load_library()
    assert [L.rt_octree_reference_bytes(s) for s in (30, 300, 3000)] == [543136, 4967896, 49215496]


def test_ppm_formatter_matches_reference_writer(pkg, O):
    rng = np.random.default_rng(3)
    fb = rng.random((13, 17, 3), dtype=np.float32)
    fb[0, 0] = (0.0, 1.0, 0.99999)
    assert pkg.format_ppm(fb) == O.write_ppm(fb)
    assert np.array_equal(pkg.quantise(fb), O.quantise(fb))


def test_no_cpu_fallback(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(pkg.RtError, match="no CPU fallback"):
        pkg.RayTracer(0)


def test_missing_library_fails_loudly(pkg, tmp_path):
    with pytest.raises(pkg.RtError, match="missing"):
        pkg.load_library(str(tmp_path / "librt_b200.so"))


def test_product_never_touches_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py may use oracle/: the package must not import, link or open it."""
    pk = os.path.join(ROOT, "dd2360-raytracing_b200")
    for dirpath, dirs, files in os.walk(pk):
        dirs[:] = [d for d in dirs if d not in ("build", "__pycache__")]
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                for banned in ("rto_", "librt_oracle", "oracle_py", "rt_oracle.h", "load_oracle", "_ref/"):
                    assert banned not in txt, (f, banned)


def test_library_skip_ahead_matches_curand(pkg, golden_dir):
    """rt_xorwow_state (host side, no GPU): the product's own skip-ahead matrices against cuRAND's answers."""
    import json
    kat = json.load(open(os.path.join(golden_dir, "curand_subsequence_kat.json")))
    for c in kat["cases"] + kat["random_cases"]:
        assert [int(x) for x in pkg.xorwow_state(c["seed"], c["subsequence"])] == c["state"], c
    with pytest.raises(pkg.RtError):
        pkg.xorwow_state(1984, 2 ** 40)


def test_experiment_harness_tables_on_cpu():
    """analysis/run_experiment.py: the summary tables (the notebook's two figures) from synthetic run rows — no GPU needed;
    also that the product scripts never reach into oracle/."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("run_experiment", os.path.join(ROOT, "analysis", "run_experiment.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    assert [mod.spheres_per_leaf(n) for n in (488, 9000, 100000, 1000000)] == [30, 30, 300, 3000]
    rows = []
    for mode, k in (("BASELINE", 4.0), ("OCTREE", 2.0)):
        for it in (1, 2, 3):
            rows.append({"mode": mode, "n": 488, "radius": 0.1, "iter": it, "spl": 30, "world_s": 1e-3, "octree_s": 2e-4, "render_s": 5e-3,
                         "kernel_ms": k + 0.1 * it, "total_s": 8e-3, "rays": 19_000_000, "mrays_s": 19_000 / (k + 0.1 * it),
                         "mem_used_mib": 640.0, "ppm": ""})
    md = mod.summarise(rows, 1200, 800, 10)
    line = [l for l in md.splitlines() if l.startswith("| 488 |")][0]
    assert "| 4.200 | 2.200 | 1.91x |" in line and "median of 3 runs" in md and "SPHERE_RADIUS = 0.1" in md
    src = open(os.path.join(ROOT, "analysis", "run_experiment.py")).read()
    assert "load_oracle" not in src and "oracle_py" not in src
