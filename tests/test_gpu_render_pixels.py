"""rt_render_pixels: a caller-given list of pixels, bit-identical to the same pixels of the full frame.

Every kernel path (FP32 lane walk, flat sweep with and without the staged geometry, flat grid, cooperative kernel with two and
four candidates per lane, forced variants, the FP16 kernel in octree and flat mode) is held to the frame it would render, for
both seedings and for final and linear values, on shuffled, partial, duplicated, out-of-range, windowed and single-pixel lists.
The full-size goldens of the reference's CUDA builds, stored as pixel subsets, are checked from their pixels alone."""
import ctypes as C
import json
import os

import numpy as np
import pytest

RT_ERR_INVALID, RT_ERR_STATE = 10001, 10002

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _frame(rt, args, finalize):
    """The whole frame as (nx*ny, 3) — rt_render (finalize) or rt_render_accumulate — and its stats."""
    import torch
    fb = torch.empty((args.ny, args.nx, 3), dtype=torch.float32, device="cuda")
    st = rt.render_device(args, fb.data_ptr()) if finalize else rt.render_accumulate(args, fb.data_ptr())
    return fb.cpu().numpy().reshape(-1, 3), st


def _lists(pkg, nx, ny, rng):
    npix = nx * ny
    sub = rng.integers(0, npix, 300)
    sub = np.concatenate([sub, sub[:40], [npix, npix + 5, 0xFFFFFFFF]]).astype(np.uint32)   # duplicates, out of the frame
    rng.shuffle(sub)
    return {
        "whole_shuffled": rng.permutation(npix).astype(np.uint32),
        "subset_dups_out_of_range": sub,
        "window": pkg.window_pixels(nx, ny, 3, nx - 5, 2, ny - 1),          # no edge on the 8x4 grid
        "single": np.array([npix // 2 + 7], np.uint32),
        "count_77": rng.integers(0, npix, 77).astype(np.uint32),
    }


# (id, spheres, SPHERES_PER_LEAF or None for the flat list, precision, variant, kernel the frame uses)
FP32, FP16 = 0, 1
CASES = [
    ("fp32_oct_488_lane", 488, 30, FP32, 0, "k_render<octree>"),
    ("fp32_oct_8000", 8000, 300, FP32, 0, "k_render<octree>"),
    ("fp32_oct_100k_coop2", 100000, 300, FP32, 0, "k_render_coop"),
    ("fp32_oct_1M_coop4", 1000000, 3000, FP32, 0, "k_render_coop"),
    ("fp32_flat_200_sweep_staged", 200, None, FP32, 0, "k_render<list>"),
    ("fp32_flat_488_grid", 488, None, FP32, 0, "k_render<octree>"),      # hitable_list::hit answered through the grid
    ("fp32_flat_20000_v20_sweep_global", 20000, None, FP32, 20, "k_render<list>"),
    ("fp32_oct_100k_v1_lane", 100000, 300, FP32, 1, "k_render<octree>"),
    ("fp32_oct_488_v31_pixel_queue", 488, 30, FP32, 31, "k_render<octree>"),
    ("fp32_oct_8000_v40_coop", 8000, 300, FP32, 40, "k_render_coop"),
    ("fp16_oct_488", 488, 30, FP16, 0, "k_render_h"),
    ("fp16_flat_488", 488, None, FP16, 0, "k_render_h"),
    ("fp16_oct_8000", 8000, 30, FP16, 0, "k_render_h"),
    ("fp16_flat_8000", 8000, None, FP16, 0, "k_render_h"),
]


# ---- CPU tier ----------------------------------------------------------------------------------------------------------------

def test_window_pixels_covers_the_rectangle_once_in_tile_order(pkg):
    nx, ny = 50, 23
    for i0, i1, j0, j1 in [(0, 50, 0, 23), (3, 45, 2, 15), (7, 8, 5, 6), (5, 21, 1, 4), (49, 50, 0, 23)]:
        w = pkg.window_pixels(nx, ny, i0, i1, j0, j1)
        assert w.dtype == np.uint32 and len(w) == (i1 - i0) * (j1 - j0)
        i, j = (w % nx).astype(np.int64), (w // nx).astype(np.int64)
        assert len(np.unique(w)) == len(w)
        assert ((i >= i0) & (i < i1) & (j >= j0) & (j < j1)).all()
        # 8x4 tiles from the rectangle's corner, row by row; pixels row by row inside a tile
        tile = (j - j0) // 4 * ((i1 - i0 + 7) // 8) + (i - i0) // 8
        key = tile * 32 + (j - j0) % 4 * 8 + (i - i0) % 8
        assert (np.diff(key) > 0).all()
    for bad in [(0, 51, 0, 1), (3, 3, 0, 1), (0, 1, 5, 2), (-1, 2, 0, 1)]:
        with pytest.raises(ValueError):
            pkg.window_pixels(nx, ny, *bad)


def test_binding_declares_rt_render_pixels(pkg):
    assert "rt_render_pixels" in pkg.ABI_SYMBOLS
    fn = pkg.load_library().rt_render_pixels
    assert fn.restype is C.c_int and len(fn.argtypes) == 7


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_pixel_lists_equal_the_frame_bit_for_bit(rt, pkg, case):
    name, n, spl, prec, variant, kernel = case
    octree = spl is not None
    rt.create_world(n, 0.1, prec)
    if octree:
        rt.build_octree(spl, prec)
    nx, ny, ns = (40, 23, 1) if n >= 1000000 else (83, 45, 2)
    lists = _lists(pkg, nx, ny, np.random.default_rng(n + variant))
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        kw = dict(seed_mode=seed, precision=prec, variant=variant)
        for finalize in (True, False):
            ref, fst = _frame(rt, rt.args(nx, ny, ns, octree, **kw), finalize)
            assert fst["kernel"].startswith(kernel), fst["kernel"]
            for lname, pix in lists.items():
                got, st = rt.render_pixels(nx, ny, ns, pix, use_octree=octree, finalize=finalize, **kw)
                inside = pix < nx * ny
                want = np.zeros((len(pix), 3), np.float32)
                want[inside] = ref[pix[inside]]
                bad = np.nonzero((_bits(got) != _bits(want)).any(axis=1))[0]
                assert len(bad) == 0, (lname, seed, finalize, int(bad[0]), int(pix[bad[0]]), got[bad[0]], want[bad[0]])
                assert st["kernel_id"] == fst["kernel_id"] and st["paths"] == ns * int(inside.sum()), (lname, st, fst)
                if lname == "whole_shuffled":
                    assert st["rays"] == fst["rays"]
                if lname == "single":              # duplicates trace their rays again: rays add up per entry
                    _, st3 = rt.render_pixels(nx, ny, ns, np.repeat(pix, 3), use_octree=octree, finalize=finalize, **kw)
                    assert st3["rays"] == 3 * st["rays"] and st3["paths"] == 3 * st["paths"]


@gpu
def test_stats_null_is_asynchronous_and_reported_afterwards(rt, pkg):
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    nx, ny, ns = 64, 32, 2
    pix = torch.from_numpy(pkg.window_pixels(nx, ny, 0, nx, 0, ny).view(np.int32)).cuda()
    out = torch.empty((pix.numel(), 3), dtype=torch.float32, device="cuda")
    assert rt.render_pixels_device(rt.args(nx, ny, ns, True), pix.data_ptr(), pix.numel(), out.data_ptr(), want_stats=False) is None
    st = rt.last_render_stats()
    ref, fst = _frame(rt, rt.args(nx, ny, ns, True), True)
    assert st["rays"] == fst["rays"] and st["paths"] == fst["paths"] and st["kernel_id"] == fst["kernel_id"]
    got = out.cpu().numpy()
    assert np.array_equal(_bits(got), _bits(ref[pix.cpu().numpy().view(np.uint32)]))


@gpu
def test_errors_write_nothing(rt, pkg):
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    nx, ny, ns, count = 40, 24, 1, 64
    pix = torch.arange(count, dtype=torch.int32, device="cuda")
    out = torch.full((count, 3), 7.0, dtype=torch.float32, device="cuda")
    host_pix = np.arange(count, dtype=np.uint32)
    host_out = np.full((count, 3), 7.0, np.float32)
    good = rt.args(nx, ny, ns, True)

    def call(r=rt, args=good, p=pix.data_ptr(), n=count, o=out.data_ptr(), finalize=1):
        return r.L.rt_render_pixels(r._ctx, C.byref(args) if args is not None else None, C.c_void_p(p), n, C.c_void_p(o), finalize, None)

    assert call(args=None) == RT_ERR_INVALID
    assert call(p=0) == RT_ERR_INVALID
    assert call(o=0) == RT_ERR_INVALID
    assert call(n=0) == RT_ERR_INVALID and call(n=-5) == RT_ERR_INVALID
    assert call(args=rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_TILES, shard_rank=0, shard_count=2)) == RT_ERR_INVALID
    assert call(args=rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2), finalize=0) == RT_ERR_INVALID
    assert call(p=host_pix.ctypes.data) == RT_ERR_INVALID               # a host list would fault the GPU
    assert call(o=host_out.ctypes.data) == RT_ERR_INVALID
    assert call(args=rt.args(0, ny, ns, True)) == RT_ERR_INVALID
    rt.build_octree(30, pkg.PREC_FP16)                                   # an octree for the other precision
    assert call() == RT_ERR_STATE
    rt.build_octree(30)
    assert call(args=rt.args(nx, ny, ns, True, precision=pkg.PREC_FP16)) == RT_ERR_STATE
    empty = pkg.RayTracer(0)
    try:
        assert call(r=empty) == RT_ERR_STATE                             # no scene
        empty.create_world(488, 0.1)
        assert call(r=empty) == RT_ERR_STATE                             # USE_OCTREE without an octree
    finally:
        empty.close()
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()) and (host_out == 7.0).all()
    assert call() == 0 and not bool((out == 7.0).all())


@gpu
def test_config3_full_size_pixels_without_the_frame(rt, pkg, O, golden_dir):
    """BASELINE config 3 (3840x2160x64, 100 k spheres, SPHERES_PER_LEAF 300) from its pixels alone: the committed 1/16 x 1/16
    subsample of the reference CUDA frame, the pixels whose closest hits are exact ties between spheres of different cells, and
    pixel (2070, 687) — total internal reflection meeting curand_uniform == 1.0 — against the oracle."""
    nx, ny, ns, n, spl = 3840, 2160, 64, 100000, 300
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C3_3840x2160x64"]
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).astype(np.uint32).reshape(-1)
    got, st = rt.render_pixels(nx, ny, ns, sub)
    assert len(sub) == 32400 and st["paths"] == len(sub) * ns
    assert np.array_equal(_bits(got.reshape(gsub.shape)), _bits(gsub))
    # ties: pixels are (i, j) with fb[j, i] (profiles/diff_full_frame.py), values the reference's as float hex
    ties = json.load(open(os.path.join(golden_dir, "ref_cuda", "C3_tie_pixels.json")))
    tp = np.array([j * nx + i for i, j in ties["pixels"]], np.uint32)
    want = np.array([[float.fromhex(h) for h in row] for row in ties["ref_gamma_f32_hex"]], np.float32)
    got, _ = rt.render_pixels(nx, ny, ns, tp)
    assert np.array_equal(_bits(got), _bits(want))
    i, j = 2070, 687
    got, _ = rt.render_pixels(nx, ny, ns, np.array([j * nx + i], np.uint32))
    assert np.isfinite(got).all()
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    ref, _, _ = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, True, spl, O.ARITH_DEVICE, window=(i, i + 1, j, j + 1)), blob)
    assert np.array_equal(_bits(got[0]), _bits(ref[j, i]))


@gpu
def test_config4_full_size_fp16_pixels_without_the_frame(rt, pkg, golden_dir):
    """BASELINE config 4 (USE_FP16, 4 spp) at full frame size: the committed 1/16 x 1/16 subsample of the reference's FP16 CUDA
    frame from those 32 400 pixels alone."""
    nx, ny, ns, n, spl = 3840, 2160, 4, 100000, 300
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C4_3840x2160x4"]
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
    rt.create_world(n, 0.1, pkg.PREC_FP16)
    rt.build_octree(spl, pkg.PREC_FP16)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).astype(np.uint32).reshape(-1)
    got, st = rt.render_pixels(nx, ny, ns, sub, precision=pkg.PREC_FP16)
    half = got.astype(np.float16)                         # half values widened to float: exact
    assert st["paths"] == len(sub) * ns and np.array_equal(half.astype(np.float32), got)
    assert np.array_equal(half.reshape(gsub.shape).view(np.uint16), gsub.view(np.uint16))
