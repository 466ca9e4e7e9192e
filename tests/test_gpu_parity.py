"""GPU tier (-m gpu): the CUDA path, called through the C ABI, against the oracle and the committed goldens.

Bars: bit-exact for the scene, the camera and the Octree blob (integer / index work and folded constants);
for frames the north-star bound is >= 99.5 % of pixels within 1/255 and PSNR >= 50 dB — this implementation is
held to the stricter "every pixel bit-identical in float32", with an allowance of 0.01 % of pixels for libdevice
powf (schlick) differing from the oracle's libm powf in the last bit."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

POWF_ALLOWANCE = 1e-4


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


def _frac_identical(a, b):
    return float((a.view(np.uint32) == b.view(np.uint32)).all(axis=2).mean())


def _psnr_u8(pkg, a, b):
    qa, qb = pkg.quantise(a).astype(float), pkg.quantise(b).astype(float)
    mse = ((qa - qb) ** 2).mean()
    return float("inf") if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


@pytest.mark.parametrize("n", [4, 5, 488, 8000, 100000])
def test_scene_generation_is_bit_exact(rt, O, n):
    rt.create_world(n, 0.1)
    sph, _ = O.create_world(n)
    assert rt.spheres().tobytes() == sph.tobytes()


@pytest.mark.parametrize("nx,ny", [(1200, 800), (240, 160), (3840, 2160), (7680, 4320), (37, 23)])
def test_camera_is_bit_exact(rt, O, golden_dir, nx, ny):
    rt.create_world(8, 0.1)
    rt.set_camera(nx, ny)
    got = rt.camera()
    assert np.array_equal(got, O.camera(nx, ny, O.ARITH_DEVICE).as_array())      # -0.0 == 0.0
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest.json")))
    key = f"{nx}x{ny}"
    if key in man["cameras"]:
        assert np.array_equal(got, np.array(man["cameras"][key], dtype=np.float32))   # the reference's own camera


@pytest.mark.parametrize("n,spl", [(488, 30), (8000, 30), (20000, 30), (9000, 7), (100000, 300), (100000, 30),
                                   (1000000, 3000)])
def test_gpu_octree_build_is_bit_exact(rt, O, golden_dir, n, spl):
    """Node numbering, AABBs, children, leaf buckets, counts: byte-identical to the serial reference build,
    including the cases where the reference drops spheres because all 8 buckets of a cell are full."""
    rt.create_world(n, 0.1)
    st = rt.build_octree(spl)
    sph, _ = O.create_world(n)
    blob, ost = O.build_octree(sph, spl)
    got = rt.export_octree()
    assert got.tobytes() == blob.tobytes()
    assert st["node_count"] == ost["node_count"] == 157
    assert st["entries"] == ost["entries"] and st["dropped_full"] == ost["dropped_full"]
    sha = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest.json")))["sha256"]
    key = f"n{n}_spl{spl}.octree"
    if key in sha:                                           # digest of the blob the reference itself built on the GPU box
        assert hashlib.sha256(got.tobytes()).hexdigest() == sha[key]


def test_octree_with_spheres_outside_the_root_box(rt, pkg, O):
    rng = np.random.default_rng(5)
    n = 3000
    sph = np.zeros(n, dtype=pkg.SPHERE_DTYPE)
    sph[0] = (0, -1000, -1, 1000, 0, 0.5, 0.5, 0.5, 0)
    for i in range(1, n):
        mat = int(rng.integers(0, 3))
        sph[i] = (rng.uniform(-14, 14), rng.uniform(-0.5, 2.6), rng.uniform(-14, 14), float(rng.choice([0.05, 0.1, 0.4, 1.2])),
                  mat, rng.random(), rng.random(), rng.random(), 1.5 if mat == 2 else 0.6 * rng.random())
    sph[99]["mat"] = -1
    rt.upload_world(sph)
    st = rt.build_octree(40)
    blob, ost = O.build_octree(sph, 40)
    assert rt.export_octree().tobytes() == blob.tobytes()
    assert st["dropped_outside"] == ost["dropped_outside"] > 0
    nx, ny, ns = 120, 80, 2
    fb, s = rt.render(nx, ny, ns, use_octree=True)
    ref, _, ctr = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, True, 40, O.ARITH_DEVICE), blob)
    assert s["rays"] == ctr["rays"]
    assert _frac_identical(fb, ref) >= 1 - POWF_ALLOWANCE


@pytest.mark.parametrize("n,spl,octree,nx,ny,ns", [
    (488, 30, False, 240, 160, 4),
    (488, 30, True, 240, 160, 4),
    (488, 30, True, 37, 23, 5),          # image not a multiple of the 8x4 tile
    (488, 30, False, 8, 4, 1),           # one tile
    (488, 30, True, 1, 1, 3),            # one pixel
    (8000, 30, True, 240, 160, 4),
    (20000, 30, True, 160, 96, 2),       # bucket overflow
    (100000, 300, True, 192, 108, 2),
    (6000, 30, False, 64, 48, 1),        # flat list staged in shared memory (96 KB)
    (20000, 30, False, 32, 24, 1),       # flat list too large for shared memory: global sweep
])
def test_render_matches_oracle(rt, pkg, O, n, spl, octree, nx, ny, ns):
    rt.create_world(n, 0.1)
    sph, _ = O.create_world(n)
    blob = None
    if octree:
        rt.build_octree(spl)
        blob, _ = O.build_octree(sph, spl)
    fb, s = rt.render(nx, ny, ns, use_octree=octree)
    ref, _, ctr = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, octree, spl, O.ARITH_DEVICE), blob)
    same = _frac_identical(fb, ref)
    assert same >= 1 - POWF_ALLOWANCE, f"only {same:.6f} of the pixels are bit-identical"
    assert abs(int(s["rays"]) - ctr["rays"]) <= max(2, int(POWF_ALLOWANCE * ctr["rays"])) and s["paths"] == nx * ny * ns
    within = float((np.abs(pkg.quantise(fb).astype(int) - O.quantise(ref).astype(int)) <= 1).all(axis=2).mean())
    assert within >= 0.995 and _psnr_u8(pkg, fb, ref) >= 50.0          # the north-star bound, for the record


def test_render_matches_reference_cuda_goldens(rt, pkg, golden_dir):
    """Frames produced on a B200 by the reference's own kernels (recompiled for sm_100)."""
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest.json")))
    for name, e in man["frames"].items():
        if not name.endswith(".npz"):
            continue
        gold = np.load(os.path.join(golden_dir, "ref_cuda", name))["fb"]
        rt.create_world(e["n"], 0.1)
        if e["use_octree"]:
            rt.build_octree(e["spl"])
        fb, _ = rt.render(e["nx"], e["ny"], e["ns"], use_octree=bool(e["use_octree"]))
        assert _frac_identical(fb, gold) == 1.0, name
    # BASELINE configs 1 and 2 at full size (1200x800, 10 spp): the reference's 8-bit image, byte for byte
    gold = np.load(os.path.join(golden_dir, "ref_cuda", "C2_1200x800x10_u8.npz"))["rgb"]
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    for octree in (False, True):
        fb, _ = rt.render(1200, 800, 10, use_octree=octree)
        assert np.array_equal(pkg.quantise(fb), gold)
        assert hashlib.sha256(fb.tobytes()).hexdigest() == man["frames"]["C2_1200x800x10"]["sha256_f32"]
    ppm = pkg.format_ppm(fb)
    assert ppm.startswith(b"P3\n1200 800\n255\n") and ppm.count(b"\n") == 3 + 1200 * 800


@pytest.mark.parametrize("n,spl,octree,nx,ny,ns", [
    (488, 30, True, 240, 160, 4),
    (488, 30, False, 96, 64, 2),
    (100000, 300, True, 192, 108, 2),    # cooperative kernel
])
def test_upstream_seeding_matches_oracle(rt, pkg, O, golden_dir, n, spl, octree, nx, ny, ns):
    """RT_SEED_UPSTREAM = curand_init(1984, pixel_index, 0) (main.cu:90): per-pixel states from the library's own
    skip-ahead kernel; frames bit-identical to the oracle, and to the reference's CUDA build patched to that line."""
    rt.create_world(n, 0.1)
    sph, _ = O.create_world(n)
    blob = None
    if octree:
        rt.build_octree(spl)
        blob, _ = O.build_octree(sph, spl)
    fb, s = rt.render(nx, ny, ns, use_octree=octree, seed_mode=pkg.SEED_UPSTREAM)
    ref, _, ctr = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE),
                           O.make_params(nx, ny, ns, octree, spl, O.ARITH_DEVICE, seed_mode=O.SEED_UPSTREAM), blob)
    assert _frac_identical(fb, ref) >= 1 - POWF_ALLOWANCE and s["launches"] == 2
    assert abs(int(s["rays"]) - ctr["rays"]) <= max(2, int(POWF_ALLOWANCE * ctr["rays"]))
    gold = os.path.join(golden_dir, "ref_cuda", f"n{n}_oct_upseed_{nx}x{ny}x{ns}.npz")
    if octree and os.path.exists(gold):
        assert _frac_identical(fb, np.load(gold)["fb"]) == 1.0


def test_upstream_seeding_spp_shards_use_disjoint_subsequences(rt, pkg):
    import torch
    nx, ny = 64, 48
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    a = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
    b = torch.zeros_like(a)
    c = torch.zeros_like(a)
    rt.render_accumulate(rt.args(nx, ny, 2, True, seed_mode=pkg.SEED_UPSTREAM), a.data_ptr())
    rt.render_accumulate(rt.args(nx, ny, 4, True, seed_mode=pkg.SEED_UPSTREAM, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2), b.data_ptr())
    rt.render_accumulate(rt.args(nx, ny, 4, True, seed_mode=pkg.SEED_UPSTREAM, shard_mode=pkg.SHARD_SPP, shard_rank=1, shard_count=2), c.data_ptr())
    assert torch.equal(a, b) and not torch.equal(b, c)


@pytest.mark.parametrize("n", [488, 6000, 20000])
def test_flat_list_grid_and_sweep_kernels_agree(rt, n):
    """USE_OCTREE off: the default answers hitable_list::hit through the grid over all spheres; variant 20 forces the
    N-tests-per-ray sweep (shared-memory staged by TMA up to ~14 k spheres, global memory above).  Same frame."""
    rt.create_world(n, 0.1)
    a, sa = rt.render(64, 40, 2, use_octree=False)
    b, sb = rt.render(64, 40, 2, use_octree=False, variant=20)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and sa["rays"] == sb["rays"]


def test_metal_fuzz_is_clamped_like_the_reference_constructor(rt, pkg):
    sph = np.zeros(8, dtype=pkg.SPHERE_DTYPE)
    sph[0] = (0, -1000, -1, 1000, 0, 0.5, 0.5, 0.5, 0)
    for i in range(1, 8):
        sph[i] = (i - 4, 0.5, 0, 0.4, 1, 0.8, 0.8, 0.8, 0.25 * i)       # fuzz 0.25 .. 1.75
    rt.upload_world(sph)
    got = rt.spheres()["param"][1:]
    assert np.array_equal(got, np.minimum(sph["param"][1:], 1.0).astype(np.float32))   # material.h:67


@pytest.mark.parametrize("n,spl", [(488, 30), (8000, 30), (100000, 300)])
def test_closest_hit_per_ray(rt, O, n, spl):
    """hitTree / hitable_list::hit for individual rays (random origins and directions, also from outside the root
    box and from below the tree): sphere index and t bit-identical to the oracle."""
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    rr = np.random.default_rng(n)
    R = 1500
    org = np.stack([rr.uniform(-13, 14, R), rr.uniform(0.02, 3, R), rr.uniform(-13, 13, R)], 1).astype(np.float32)
    dirs = rr.normal(size=(R, 3)).astype(np.float32)
    dirs[:50, 1] = 0.0                                                # axis-parallel components: division by zero paths
    dirs[50:80, 0] = 0.0
    gi, gt = rt.trace_rays(org, dirs, True)
    hits = 0
    for k in range(R):
        oi, ot = O.closest_hit(sph, org[k], dirs[k], blob, spl, True)
        assert oi == gi[k] and (oi < 0 or np.float32(ot) == gt[k]), (k, oi, ot, gi[k], gt[k])
        hits += oi >= 0
    assert 0.2 * R < hits < R
    if n <= 8000:
        bi, bt = rt.trace_rays(org, dirs, False)
        for k in range(0, R, 3):
            oi, ot = O.closest_hit(sph, org[k], dirs[k], None, spl, False)
            assert oi == bi[k] and (oi < 0 or np.float32(ot) == bt[k])


def test_full_size_properties_config3(rt, pkg):
    """BASELINE config 3 scene (100k spheres, SPL 300) at 3840x2160: properties that need no oracle run —
    determinism, tile shards summing to the unsharded frame bit for bit, spp shards preserving the sample count."""
    import torch
    nx, ny, ns = 3840, 2160, 2
    rt.create_world(100000, 0.1)
    rt.build_octree(300)
    a = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
    b = torch.zeros_like(a)
    acc = torch.zeros_like(a)
    s1 = rt.render_accumulate(rt.args(nx, ny, ns, True), a.data_ptr())
    s2 = rt.render_accumulate(rt.args(nx, ny, ns, True), b.data_ptr())
    assert torch.equal(a, b) and s1["rays"] == s2["rays"] and s1["paths"] == nx * ny * ns
    assert bool(torch.isfinite(a).all()) and float(a.min()) >= 0.0
    rays = 0
    for g in range(3):
        part = torch.empty_like(a)
        st = rt.render_accumulate(rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_TILES, shard_rank=g, shard_count=3), part.data_ptr())
        rays += st["rays"]
        acc += part
    assert torch.equal(acc, a) and rays == s1["rays"]
    paths = 0
    for g in range(2):
        st = rt.render_accumulate(rt.args(nx, ny, 3, True, shard_mode=pkg.SHARD_SPP, shard_rank=g, shard_count=2), b.data_ptr())
        paths += st["paths"]
    assert paths == nx * ny * 3
    fb = torch.empty_like(a)
    rt.finalize(a.data_ptr(), fb.data_ptr(), nx, ny, ns)
    rt.synchronize()
    want = torch.sqrt(a * np.float32(1.0 / ns))
    assert torch.equal(fb, want)


def test_octree_and_flat_list_agree_at_488(rt):
    """Host brute == host octree bit for bit in the reference (SURVEY A.4); the same must hold here."""
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    a, sa = rt.render(300, 200, 6, use_octree=True)
    b, sb = rt.render(300, 200, 6, use_octree=False)
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and sa["rays"] == sb["rays"]


def test_spp_shard_zero_is_the_reference_stream(rt, pkg):
    import torch
    nx, ny = 96, 64
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    full = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
    sh0 = torch.zeros_like(full)
    rt.render_accumulate(rt.args(nx, ny, 3, True), full.data_ptr())
    rt.render_accumulate(rt.args(nx, ny, 6, True, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2), sh0.data_ptr())
    assert torch.equal(full, sh0)          # shard 0 of a 6-spp frame = the first 3 samples of the reference stream


def test_error_behaviour(rt, pkg):
    fresh = pkg.RayTracer(0)
    with pytest.raises(pkg.RtError, match="no scene"):
        fresh.render(8, 8, 1, use_octree=False)
    fresh.create_world(16, 0.1)
    with pytest.raises(pkg.RtError, match="no octree"):
        fresh.render(8, 8, 1, use_octree=True)
    with pytest.raises(pkg.RtError):
        fresh.create_world(3, 0.1)
    with pytest.raises(pkg.RtError, match="seed_mode"):
        fresh.render(8, 8, 1, use_octree=False, seed_mode=7)
    fresh.close()


# ---- USE_FP16 (BASELINE config 4) --------------------------------------------------------------------------------------
# The reference built with -DUSE_FP16 renders a structurally different image (no ground plane: r*r overflows half,
# SURVEY D9), so the bar is stated against the REFERENCE'S OWN FP16 CUDA build on a B200 (tests/golden/ref_cuda/*fp16*),
# not against FP32.  The product re-states that build's arithmetic operation by operation with the same intrinsics
# (rt_half.cuh); what can still differ is where ptxas fuses a half multiply-add differently in the two programs, which
# flips a rejection-sampling or hit decision and re-rolls that pixel (refract's last line is such a place: FP32 fuses its
# right product, FP16 its left).  Stated bounds: scene, camera and leaf lists bit-exact; >= 99.9 % of pixels bit-identical
# and PSNR >= 50 dB on the 8-bit image per golden frame.  Measured on B200: 100 % identical on all four golden frames.
FP16_MIN_IDENTICAL = 0.999
FP16_MIN_PSNR = 50.0


def _morton(ix, iy, iz):
    m = 0
    for b in (2, 1, 0):
        m = (m << 3) | (((ix >> b) & 1) << 2) | (((iy >> b) & 1) << 1) | ((iz >> b) & 1)
    return m


def test_fp16_scene_is_bit_exact(rt, pkg, O, golden_dir):
    """create_world of the FP16 build: the scene dumped from the reference's own kernel on a B200."""
    gold = np.load(os.path.join(golden_dir, "ref_cuda", "n488_fp16_spheres.npy"))
    rt.create_world(488, 0.1, precision=pkg.PREC_FP16)
    assert rt.spheres().tobytes() == gold.tobytes()
    if O.RefHost.available("oct_spl30_fp16"):            # the reference's own FP16 create_world body, host-compiled
        for n in (8000, 20000):
            rh = O.RefHost("oct_spl30_fp16").create_world(n, 0.1, 64, 48)
            rt.create_world(n, 0.1, precision=pkg.PREC_FP16)
            assert rt.spheres().tobytes() == rh.spheres().tobytes(), n
            rh.destroy()


def test_fp16_camera_is_bit_exact(rt, golden_dir):
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest.json")))
    rt.create_world(8, 0.1)
    for key, want in man["cameras_fp16"].items():
        nx, ny = (int(v) for v in key.split("x"))
        rt.set_camera(nx, ny)
        assert np.array_equal(rt.camera_half(nx, ny), np.array(want, dtype=np.float32)), key


@pytest.mark.parametrize("n,spl", [(488, 30), (8000, 30)])
def test_fp16_octree_leaf_lists_match_reference(rt, pkg, golden_dir, n, spl):
    """The sphere lists of every level-3 node of the Octree the reference's FP16 build constructs (half-rounded centres
    against half-rounded grown bounds), cell by cell."""
    gold = np.load(os.path.join(golden_dir, "ref_cuda", f"n{n}_spl{spl}_fp16_cells.npz"))
    rt.create_world(n, 0.1, precision=pkg.PREC_FP16)
    rt.build_octree(spl, precision=pkg.PREC_FP16)
    t = rt.debug_tree()
    cs = t["cell_start"].view(np.uint32)
    cl = t["cell_list"].view(np.uint32)
    seen = 0
    for k, low in enumerate(gold["low"]):
        ix, iy, iz = int(round((low[0] + 11) / 2.75)), int(round(low[1] / 0.25)), int(round((low[2] + 11) / 2.75))
        m = _morton(ix, iy, iz)
        want = gold["idx"][gold["start"][k]:gold["start"][k + 1]]
        got = cl[cs[m]:min(cs[m + 1], cs[m] + 8 * spl)]
        assert np.array_equal(got.astype(np.int64), want.astype(np.int64)), (k, low)
        seen += 1
    assert seen == int((np.diff(cs.astype(np.int64)) > 0).sum())          # no cell the reference does not have


def test_fp16_frames_match_reference_fp16_build(rt, pkg, golden_dir):
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest.json")))
    report = {}
    for name, e in man["extra_frames"].items():
        if not e.get("fp16"):
            continue
        gold = np.load(os.path.join(golden_dir, "ref_cuda", name))["fb"].astype(np.float32)
        rt.create_world(e["n"], 0.1, precision=pkg.PREC_FP16)
        if e["use_octree"]:
            rt.build_octree(e["spl"], precision=pkg.PREC_FP16)
        fb, st = rt.render(e["nx"], e["ny"], e["ns"], use_octree=bool(e["use_octree"]), precision=pkg.PREC_FP16)
        same = float((fb == gold).all(axis=2).mean())
        report[name] = (same, _psnr_u8(pkg, np.nan_to_num(fb), np.nan_to_num(gold)), st["rays"] / st["paths"])
    print("FP16 vs reference FP16 build (identical pixels, PSNR dB, rays/path):", report)
    assert report
    for name, (same, psnr, _) in report.items():
        assert same >= FP16_MIN_IDENTICAL and psnr >= FP16_MIN_PSNR, (name, same, psnr)


def test_fp16_octree_and_flat_list_agree(rt, pkg):
    """As in FP32, the tree only restricts which spheres are tested; with 488 spheres nothing is dropped, so both modes
    must produce the same half image (ties included: same test order)."""
    rt.create_world(488, 0.1, precision=pkg.PREC_FP16)
    rt.build_octree(30, precision=pkg.PREC_FP16)
    a, sa = rt.render(200, 120, 3, use_octree=True, precision=pkg.PREC_FP16)
    b, sb = rt.render(200, 120, 3, use_octree=False, precision=pkg.PREC_FP16)
    print("fp16 tree vs list identical:", float((a == b).all(axis=2).mean()), sa["rays"], sb["rays"])
    with pytest.raises(pkg.RtError, match="precision"):
        rt.render(8, 8, 1, use_octree=True)                                # FP32 render on an FP16 tree


def test_dropin_class_surface_renders_the_same_frame(rt, pkg, O, tmp_path):
    """include/rt_dropin.h end to end: a C++ program builds the world with sphere / hitable_list / materials / camera,
    uploads it through rt_upload_world + rt_apply_camera and renders; same frame as the generated scene."""
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe, out = str(tmp_path / "render_dropin"), str(tmp_path / "fb.bin")
    lib_dir = os.path.dirname(pkg.LIB_PATH)
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "dropin", "render_dropin.cpp"),
                    "-o", exe, f"-L{lib_dir}", "-lrt_b200", f"-Wl,-rpath,{lib_dir}"], check=True)
    sph, _ = O.create_world(488)
    lines = [str(len(sph))] + [" ".join([float(s["cx"]).hex(), float(s["cy"]).hex(), float(s["cz"]).hex(), float(s["radius"]).hex(),
                                         str(int(s["mat"])), float(s["ax"]).hex(), float(s["ay"]).hex(), float(s["az"]).hex(),
                                         float(s["param"]).hex()]) for s in sph]
    subprocess.run([exe, out], input="\n".join(lines) + "\n", text=True, check=True)
    got = np.fromfile(out, dtype=np.float32).reshape(48, 64, 3)
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    want, _ = rt.render(64, 48, 2, use_octree=True)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_experiment_harness_sweep(tmp_path):
    """analysis/run_experiment.py (the reference's run_experiment.sh + notebook tables): a 2-size sweep writes runs.csv,
    summary.md and a PPM per run in the reference's naming; BASELINE and OCTREE trace the same rays."""
    import csv
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = str(tmp_path / "experiments")
    subprocess.run([sys.executable, os.path.join(root, "analysis", "run_experiment.py"), "--sizes", "488,2000", "--radii", "0.1", "--iters", "2",
                    "--nx", "120", "--ny", "80", "--ns", "2", "--out", out, "--ppm"], check=True, stdout=subprocess.DEVNULL)
    rows = list(csv.DictReader(open(os.path.join(out, "runs.csv"))))
    assert len(rows) == 2 * 2 * 2 and all(float(r["kernel_ms"]) > 0 for r in rows)
    by = {(r["mode"], r["n"], r["iter"]): r for r in rows}
    assert by[("BASELINE", "488", "1")]["rays"] == by[("OCTREE", "488", "1")]["rays"]
    assert open(by[("OCTREE", "2000", "2")]["ppm"], "rb").read(3) == b"P3\n"
    assert "octree speed-up" in open(os.path.join(out, "summary.md")).read()


def test_device_ppm_writer_matches_host_writer_byte_for_byte(rt, pkg):
    """csrc/rt_ppm.cu against rt_format_ppm (itself pinned on the reference's writer): rendered frames, odd sizes, and
    values the quantiser must treat like the x86 cast does (negative, > 1, huge, inf, NaN)."""
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    txt, st = rt.render_ppm(203, 117, 2, use_octree=True)
    fb, _ = rt.render(203, 117, 2, use_octree=True)
    assert txt == pkg.format_ppm(fb) and txt.startswith(b"P3\n203 117\n255\n") and st["rays"] > 0
    rng = np.random.default_rng(7)
    for nx, ny in [(1, 1), (7, 3), (256, 1), (257, 5), (1200, 800), (33, 1031)]:
        fb = rng.random((ny, nx, 3), dtype=np.float32)
        flat = fb.reshape(-1)
        k = min(flat.size, 12)
        flat[:k] = np.array([0.0, 1.0, -0.5, 3.7, 1e4, -1e6, 8388607.0, 1e12, -1e30, np.inf, -np.inf, np.nan], dtype=np.float32)[:k]
        dev = torch.from_numpy(fb).cuda()
        assert rt.format_ppm_device(dev.data_ptr(), nx, ny) == pkg.format_ppm(fb), (nx, ny)


def test_cli_modes_write_the_reference_image(pkg, golden_dir, tmp_path):
    """`RayTracing [mode]` (main.cu:347-477) at BASELINE config 2: mode 3 writes output.ppm, mode 0 the same bytes to stdout,
    mode 1 nothing; the pixels are the reference CUDA build's 8-bit image; a non-numeric mode throws like std::stoi."""
    import subprocess
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "RayTracing")
    env = dict(os.environ, RT_NUM_SPHERES="488", RT_SPHERES_PER_LEAF="30")
    r3 = subprocess.run([exe, "3"], cwd=tmp_path, env=env, capture_output=True, check=True)
    ppm = (tmp_path / "output.ppm").read_bytes()
    assert r3.stdout == b"" and b"took " in r3.stderr and b"Number of spheres: 488" in r3.stderr
    tok = ppm.split()
    assert tok[:4] == [b"P3", b"1200", b"800", b"255"]
    rgb = np.array(tok[4:], dtype=np.int64).reshape(800, 1200, 3)
    gold = np.load(os.path.join(golden_dir, "ref_cuda", "C2_1200x800x10_u8.npz"))["rgb"]
    assert np.array_equal(rgb, gold)
    r0 = subprocess.run([exe], cwd=tmp_path, env=env, capture_output=True, check=True)
    assert r0.stdout == ppm
    (tmp_path / "output.ppm").unlink()
    r1 = subprocess.run([exe, "1"], cwd=tmp_path, env=env, capture_output=True, check=True)
    assert r1.stdout == b"" and not (tmp_path / "output.ppm").exists()
    assert subprocess.run([exe, "x"], cwd=tmp_path, env=env, capture_output=True).returncode != 0


@pytest.mark.parametrize("n,spl,nx,ny,ns", [
    (100000, 300, 192, 108, 2),
    (8000, 30, 240, 160, 4),
    (20000, 30, 160, 96, 2),             # bucket overflow: no_drops = 0, every hit goes through the exact visibility rule
    (488, 30, 37, 23, 5),                # big spheres in the prolog list, image not a multiple of the tile
])
def test_pooled_kernel_matches_oracle(rt, O, n, spl, nx, ny, ns):
    """The scenes that held the retired pooled kernel to the oracle, rendered by k_render_coop forced (variant 40; the automatic
    choice takes it from 40 k spheres on)."""
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    fb, s = rt.render(nx, ny, ns, use_octree=True, variant=40)
    ref, _, ctr = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, True, spl, O.ARITH_DEVICE), blob)
    assert _frac_identical(fb, ref) >= 1 - POWF_ALLOWANCE
    assert abs(int(s["rays"]) - ctr["rays"]) <= max(2, int(POWF_ALLOWANCE * ctr["rays"])) and s["paths"] == nx * ny * ns


def test_pooled_and_plain_kernels_agree_at_4k(rt):
    """Config 3 scene at 3840x2160 (tile claims per warp, single-pixel claims with variant 31): the same frame from
    k_render_coop (variant 40, in place of the retired pooled kernel), k_render (variant 1) and the pixel queue."""
    import torch
    nx, ny = 3840, 2160
    rt.create_world(100000, 0.1)
    rt.build_octree(300)
    fbs = []
    for v in (40, 1, 31):
        fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        st = rt.render_device(rt.args(nx, ny, 1, True, variant=v), fb.data_ptr())
        fbs.append((fb, st["rays"]))
    assert torch.equal(fbs[0][0], fbs[1][0]) and torch.equal(fbs[0][0], fbs[2][0]) and fbs[0][1] == fbs[1][1] == fbs[2][1]


def test_config3_full_size_frame_is_the_reference_cuda_frame(rt, pkg, O, golden_dir):
    """BASELINE config 3 at FULL size (3840x2160, 64 spp, 1.04e9 rays) against the frame the reference's own CUDA build wrote
    on a B200 (tests/golden/gen_ref_cuda_full.sh; 178 s there): sha256 of the float framebuffer and of the integer PPM values,
    and the committed 1/16 x 1/16 subsample pixel by pixel.  Two things this pins that small frames never reach:
    * exact ties between DIFFERENT spheres (bit-identical t; ~170 pixels of this frame): the reference keeps the sphere with the
      smaller index (same level-3 cell, leaf lists in ascending order);
    * pixel (2070, 687), sample 36: total internal reflection meets curand_uniform == 1.0, the reference reads its uninitialised
      `refracted` (material.h:88,109) — the value its sm_100 build has there is reproduced (rt_shade.cuh), so the pixel is finite as
      in the reference's frame (with zeros it would be NaN).  The oracle's window around it agrees bit for bit."""
    import sys
    import torch
    sys.path.insert(0, golden_dir)
    from digest_frame import digest, subsample16
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C3_3840x2160x64"]
    nx, ny, ns, n, spl = 3840, 2160, 64, 100000, 300
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    st = rt.render_device(rt.args(nx, ny, ns, True), fb.data_ptr())
    frame = fb.cpu().numpy()
    assert torch.isfinite(fb).all() and st["paths"] == nx * ny * ns
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
    assert np.array_equal(subsample16(frame).view(np.uint32), gsub.view(np.uint32))
    d = digest(frame)
    assert d["sha256_raw"] == man["sha256_raw"], (d, st)
    assert d["sha256_i32_ppm_order"] == man["sha256_i32_ppm_order"]
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    i0, i1, j = 2064, 2077, 687
    ref, _, _ = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, True, spl, O.ARITH_DEVICE, window=(i0, i1, j, j + 1)), blob)
    assert np.array_equal(frame[j, i0:i1].view(np.uint32), ref[j, i0:i1].view(np.uint32))


def test_config4_full_size_4spp_frame_is_the_reference_fp16_frame(rt, pkg, golden_dir):
    """BASELINE config 4 (USE_FP16) at full frame size, 4 spp — the sample count at which the reference's FP16 CUDA build was run on a
    B200 (3.4 s there; tests/golden/gen_ref_cuda_full.sh): sha256 of the half framebuffer and of the integer PPM values, plus the
    committed 1/16 x 1/16 subsample pixel by pixel."""
    import sys
    import torch
    sys.path.insert(0, golden_dir)
    from digest_frame import digest, subsample16
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C4_3840x2160x4"]
    nx, ny, ns, n, spl = 3840, 2160, 4, 100000, 300
    try:
        rt.create_world(n, 0.1, pkg.PREC_FP16)
        rt.build_octree(spl, pkg.PREC_FP16)
        fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        st = rt.render_device(rt.args(nx, ny, ns, True, precision=pkg.PREC_FP16), fb.data_ptr())
        frame = fb.cpu().numpy().astype(np.float16)              # the frame holds half values widened to float: exact
        assert st["paths"] == nx * ny * ns and np.array_equal(frame.astype(np.float32), fb.cpu().numpy())
        gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
        assert np.array_equal(subsample16(frame).view(np.uint16), gsub.view(np.uint16))
        d = digest(frame)
        assert d["sha256_raw"] == man["sha256_raw"], d
        assert d["sha256_i32_ppm_order"] == man["sha256_i32_ppm_order"]
    finally:
        rt.create_world(488, 0.1)                                 # leave the shared context in FP32
        rt.build_octree(30)


def test_one_million_spheres_default_kernel_matches_oracle(rt, pkg, O):
    """BASELINE config 5's scene (1 M spheres, SPHERES_PER_LEAF 3000) through the AUTOMATIC kernel choice (the warp-cooperative
    kernel, four candidates per lane at this list length): a small frame and a window of the 8K frame against the oracle, and
    individual closest hits (sphere index and t) for random rays."""
    n, spl = 1000000, 3000
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    fb, s = rt.render(96, 54, 2, use_octree=True)
    assert s["kernel"].startswith("k_render_coop")
    ref, _, ctr = O.render(sph, O.camera(96, 54, O.ARITH_DEVICE), O.make_params(96, 54, 2, True, spl, O.ARITH_DEVICE), blob)
    assert _frac_identical(fb, ref) >= 1 - POWF_ALLOWANCE and abs(int(s["rays"]) - ctr["rays"]) <= 2
    # a window of the full 7680x4320 frame (camera rays of the real configuration: a finer pixel grid over the same carpet)
    import torch
    nx, ny, ns = 7680, 4320, 1
    big = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    rt.render_device(rt.args(nx, ny, ns, True), big.data_ptr())
    i0, i1, j0, j1 = 3800, 3864, 1500, 1508
    ref, _, _ = O.render(sph, O.camera(nx, ny, O.ARITH_DEVICE), O.make_params(nx, ny, ns, True, spl, O.ARITH_DEVICE, window=(i0, i1, j0, j1)), blob)
    got = big[j0:j1, i0:i1].cpu().numpy()
    assert _frac_identical(got, ref[j0:j1, i0:i1]) >= 1 - 2.0 / got[..., 0].size
    # per-ray closest hits
    rr = np.random.default_rng(5)
    R = 600
    org = np.stack([rr.uniform(-12, 13, R), rr.uniform(0.02, 2.5, R), rr.uniform(-12, 12, R)], 1).astype(np.float32)
    dirs = rr.normal(size=(R, 3)).astype(np.float32)
    gi, gt = rt.trace_rays(org, dirs, True)
    for k in range(R):
        oi, ot = O.closest_hit(sph, org[k], dirs[k], blob, spl, True)
        assert oi == gi[k] and (oi < 0 or np.float32(ot) == gt[k]), (k, oi, ot, gi[k], gt[k])
