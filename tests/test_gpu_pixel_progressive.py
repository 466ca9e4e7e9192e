"""rt_render_pixels_progressive and rt_finalize_counts: more samples for the listed pixels of a progressive frame, and the frame
finalised from per-pixel sample counts.

Every kernel path (FP32 lane walk, flat sweep with and without the staged geometry, flat grid, cooperative kernel with two and
four candidates per lane, forced variants, the FP16 kernel in octree and flat mode) is held, for both seedings, to one-shot
renders: whatever schedule of frame and list calls gives a pixel S samples leaves its sum and stream state bit for bit as one
S-sample progressive render does, and its finalised value as rt_render(ns = S).  The full-size goldens of the reference's CUDA
builds are rebuilt from their pixels in several list calls."""
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


def _dev(a):
    """A host uint32 / float32 array on the GPU (uint32 as the same 32-bit patterns in an int32 tensor)."""
    import torch
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a.copy()).cuda()


def _host(t, dtype=np.float32):
    return t.cpu().numpy().view(dtype)


class Buffers:
    """The caller's frame-indexed progressive buffers: accum (nx*ny*3 floats), stream states (nx*ny*6 words), counts (nx*ny)."""

    def __init__(self, nx, ny):
        import torch
        self.npix = nx * ny
        self.accum = torch.zeros(self.npix * 3, dtype=torch.float32, device="cuda")
        self.state = torch.zeros(self.npix * 6, dtype=torch.int32, device="cuda")
        self.counts = torch.zeros(self.npix, dtype=torch.int32, device="cuda")

    def host(self):
        return (_host(self.accum).reshape(-1, 3), _host(self.state, np.uint32).reshape(-1, 6), _host(self.counts, np.uint32))


def _frame_call(rt, args, b, first):
    return rt.render_progressive(args, b.accum.data_ptr(), b.state.data_ptr(), first)


def _list_call(rt, args, b, pix_dev, first, counts=True, want_stats=True):
    return rt.render_pixels_progressive(args, pix_dev.data_ptr(), pix_dev.numel(), b.accum.data_ptr(), b.state.data_ptr(),
                                        b.counts.data_ptr() if counts else 0, first, want_stats)


def _oneshot(rt, nx, ny, S, octree, kw):
    """(linear sums, stream states, rt_render frame) of one S-sample render, each (npix, ...)."""
    import torch
    b = Buffers(nx, ny)
    _frame_call(rt, rt.args(nx, ny, S, octree, **kw), b, True)
    fb = torch.empty(nx * ny * 3, dtype=torch.float32, device="cuda")
    rt.render_device(rt.args(nx, ny, S, octree, **kw), fb.data_ptr())
    acc, st, _ = b.host()
    return acc, st, _host(fb).reshape(-1, 3)


def _check_against_oneshots(rt, nx, ny, octree, kw, b, totals, prec, what):
    """Every pixel's sum and state equal the one-shot progressive render at its total, finalise_counts equals rt_render there,
    and the library's counts equal the host's totals."""
    import torch
    acc, st, cnt = b.host()
    assert np.array_equal(cnt, totals), what
    fb = torch.empty(nx * ny * 3, dtype=torch.float32, device="cuda")
    rt.finalize_counts(b.accum.data_ptr(), b.counts.data_ptr(), fb.data_ptr(), nx * ny, prec)
    fb = _host(fb).reshape(-1, 3)
    for S in np.unique(totals):
        ref_acc, ref_st, ref_fb = _oneshot(rt, nx, ny, int(S), octree, kw)
        m = totals == S
        for name, got, want in (("accum", _bits(acc[m]), _bits(ref_acc[m])), ("state", st[m], ref_st[m]),
                                ("finalize_counts", _bits(fb[m]), _bits(ref_fb[m]))):
            bad = np.nonzero((got != want).any(axis=1))[0]
            assert len(bad) == 0, (what, name, int(S), int(np.nonzero(m)[0][bad[0]]))


# (id, spheres, SPHERES_PER_LEAF or None for the flat list, precision, variant, kernel the frame uses) — test_gpu_render_pixels' cases
FP32, FP16 = 0, 1
CASES = [
    ("fp32_oct_488_lane", 488, 30, FP32, 0, "k_render<octree>"),
    ("fp32_oct_8000", 8000, 300, FP32, 0, "k_render<octree>"),
    ("fp32_oct_100k_coop2", 100000, 300, FP32, 0, "k_render_coop"),
    ("fp32_oct_1M_coop4", 1000000, 3000, FP32, 0, "k_render_coop"),
    ("fp32_flat_200_sweep_staged", 200, None, FP32, 0, "k_render<list>"),
    ("fp32_flat_488_grid", 488, None, FP32, 0, "k_render<octree>"),
    ("fp32_flat_20000_v20_sweep_global", 20000, None, FP32, 20, "k_render<list>"),
    ("fp32_oct_100k_v1_lane", 100000, 300, FP32, 1, "k_render<octree>"),
    ("fp32_oct_488_v31_pixel_queue", 488, 30, FP32, 31, "k_render<octree>"),
    ("fp32_oct_8000_v40_coop", 8000, 300, FP32, 40, "k_render_coop"),
    ("fp16_oct_488", 488, 30, FP16, 0, "k_render_h"),
    ("fp16_flat_488", 488, None, FP16, 0, "k_render_h"),
    ("fp16_oct_8000", 8000, 30, FP16, 0, "k_render_h"),
    ("fp16_flat_8000", 8000, None, FP16, 0, "k_render_h"),
]


def _scene(rt, n, spl, prec):
    rt.create_world(n, 0.1, prec)
    if spl is not None:
        rt.build_octree(spl, prec)
    return (40, 23) if n >= 1000000 else (83, 45)


# ---- CPU tier ----------------------------------------------------------------------------------------------------------------

def test_binding_declares_both_entry_points(pkg):
    L = pkg.load_library()
    assert "rt_render_pixels_progressive" in pkg.ABI_SYMBOLS and "rt_finalize_counts" in pkg.ABI_SYMBOLS
    vp, i32 = C.c_void_p, C.c_int
    fn = L.rt_render_pixels_progressive
    assert fn.restype is i32
    assert fn.argtypes == [vp, C.POINTER(pkg.RenderArgs), vp, i32, vp, vp, vp, i32, C.POINTER(pkg.RenderStats)]
    fn = L.rt_finalize_counts
    assert fn.restype is i32 and fn.argtypes == [vp, vp, vp, vp, C.c_size_t, i32]


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_schedules_equal_one_shot_renders(rt, pkg, case):
    """A frame call, list calls on shuffled subsets with duplicates and out-of-frame entries, a window and a single pixel with
    varied ns, then another frame call: every pixel ends where one render of its total sample count does."""
    name, n, spl, prec, variant, kernel = case
    octree = spl is not None
    nx, ny = _scene(rt, n, spl, prec)
    npix = nx * ny
    rng = np.random.default_rng(n + variant)
    sub = rng.integers(0, npix, npix // 3)
    sub = np.concatenate([sub, sub[:40], sub[:5], [npix, npix + 5, 0xFFFFFFFF]]).astype(np.uint32)
    rng.shuffle(sub)
    window = pkg.window_pixels(nx, ny, 3, nx - 5, 2, ny - 1)
    single = np.array([npix // 2 + 7], np.uint32)
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        kw = dict(seed_mode=seed, precision=prec, variant=variant)
        b = Buffers(nx, ny)
        totals = np.zeros(npix, np.uint32)
        st = _frame_call(rt, rt.args(nx, ny, 2, octree, **kw), b, True)
        assert st["kernel"].startswith(kernel), st["kernel"]
        totals += 2
        b.counts.fill_(2)                                    # rt_render_progressive keeps no counts: the caller does
        for pix, ns in ((sub, 3), (window, 1), (single, 2)):
            lst = _list_call(rt, rt.args(nx, ny, ns, octree, **kw), b, _dev(pix), False)
            inside = np.unique(pix[pix < npix])
            totals[inside] += ns
            assert lst["kernel_id"] == st["kernel_id"] and lst["paths"] == ns * len(inside), (lst, st)
            assert lst["launches"] == 2
        _frame_call(rt, rt.args(nx, ny, 1, octree, **kw), b, False)
        totals += 1
        b.counts.add_(1)
        assert len(np.unique(totals)) <= 8
        _check_against_oneshots(rt, nx, ny, octree, kw, b, totals, prec, (name, seed))


LIST_FIRST_CASES = [c for c in CASES if c[0] in ("fp32_oct_488_lane", "fp32_oct_100k_coop2", "fp32_flat_200_sweep_staged",
                                                   "fp32_flat_488_grid", "fp16_oct_488", "fp16_flat_488")]


@gpu
@pytest.mark.parametrize("case", LIST_FIRST_CASES, ids=[c[0] for c in LIST_FIRST_CASES])
def test_list_first_then_frame_calls(rt, pkg, case):
    """A first list call over the whole frame in shuffled order starts the frame's buffers; frame calls continue them."""
    name, n, spl, prec, variant, _ = case
    octree = spl is not None
    nx, ny = _scene(rt, n, spl, prec)
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        kw = dict(seed_mode=seed, precision=prec, variant=variant)
        b = Buffers(nx, ny)
        perm = np.random.default_rng(5).permutation(nx * ny).astype(np.uint32)
        _list_call(rt, rt.args(nx, ny, 2, octree, **kw), b, _dev(perm), True)
        _frame_call(rt, rt.args(nx, ny, 1, octree, **kw), b, False)
        _frame_call(rt, rt.args(nx, ny, 3, octree, **kw), b, False)
        b.counts.add_(4)
        _check_against_oneshots(rt, nx, ny, octree, kw, b, np.full(nx * ny, 6, np.uint32), prec, (name, seed))


@gpu
@pytest.mark.parametrize("prec", [FP32, FP16], ids=["fp32", "fp16"])
def test_unlisted_pixels_are_untouched(rt, pkg, prec):
    """Sentinel bit patterns in all three buffers survive everywhere except at the listed pixels inside the frame."""
    import torch
    nx, ny = _scene(rt, 488, 30, prec)
    npix = nx * ny
    b = Buffers(nx, ny)
    b.accum.view(torch.int32).fill_(0x7FA5A5A5)           # a NaN pattern: compared as bits
    b.state.fill_(-0x5A5A5A5B)
    b.counts.fill_(0x13579BD)
    rng = np.random.default_rng(11)
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        for first, ns in ((True, 2), (False, 1)):
            pix = np.concatenate([rng.integers(0, npix, 200), [npix, npix + 1, 0xFFFFFFFF]]).astype(np.uint32)
            rng.shuffle(pix)
            a0, s0, c0 = b.host()
            _list_call(rt, rt.args(nx, ny, ns, True, seed_mode=seed, precision=prec), b, _dev(pix), first)
            a1, s1, c1 = b.host()
            listed = np.zeros(npix, bool)
            listed[pix[pix < npix]] = True
            assert np.array_equal(_bits(a1[~listed]), _bits(a0[~listed]))
            assert np.array_equal(s1[~listed], s0[~listed]) and np.array_equal(c1[~listed], c0[~listed])
            assert (c1[listed] == (ns if first else c0[listed] + ns)).all()
            assert (s1[listed] != s0[listed]).any(axis=1).all()


@gpu
def test_dedupe_and_stats(rt, pkg):
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    nx, ny, ns = 64, 32, 3
    args = rt.args(nx, ny, ns, True)
    one = np.array([nx * ny // 2 + 9], np.uint32)
    st1 = _list_call(rt, args, Buffers(nx, ny), _dev(one), True)
    b3 = Buffers(nx, ny)
    st3 = _list_call(rt, args, b3, _dev(np.repeat(one, 3)), True)
    assert st3["rays"] == st1["rays"] and st3["paths"] == st1["paths"] == ns          # rt_render_pixels would trace it 3 times
    assert int(_host(b3.counts, np.uint32)[one[0]]) == ns
    _, stp = rt.render_pixels(nx, ny, ns, np.repeat(one, 3))
    assert stp["rays"] == 3 * st1["rays"]
    # the whole frame as a list in tile order: the frame call's rays and kernel
    tiles = _dev(pkg.window_pixels(nx, ny, 0, nx, 0, ny))
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        a = rt.args(nx, ny, ns, True, seed_mode=seed)
        fst = _frame_call(rt, a, Buffers(nx, ny), True)
        b = Buffers(nx, ny)
        assert _list_call(rt, a, b, tiles, True, want_stats=False) is None            # stats = NULL: asynchronous
        lst = rt.last_render_stats()
        assert lst["rays"] == fst["rays"] and lst["paths"] == fst["paths"] and lst["kernel_id"] == fst["kernel_id"]
        assert lst["launches"] == 2
        acc, _, _ = b.host()
        ref, _, _ = _oneshot(rt, nx, ny, ns, True, dict(seed_mode=seed))
        assert np.array_equal(_bits(acc), _bits(ref))
    torch.cuda.synchronize()


@gpu
def test_errors_write_nothing(rt, pkg):
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    nx, ny, ns, count = 40, 24, 1, 64
    npix = nx * ny
    pix = torch.arange(count, dtype=torch.int32, device="cuda")
    b = Buffers(nx, ny)
    b.accum.fill_(7.0); b.state.fill_(7); b.counts.fill_(7)
    host_pix = np.arange(count, dtype=np.uint32)
    host_acc = np.full(npix * 3, 7.0, np.float32)
    host_st = np.full(npix * 6, 7, np.uint32)
    host_cnt = np.full(npix, 7, np.uint32)
    good = rt.args(nx, ny, ns, True)

    def call(r=rt, args=good, p=pix.data_ptr(), n=count, a=b.accum.data_ptr(), s=b.state.data_ptr(), c=b.counts.data_ptr(), first=1):
        return r.L.rt_render_pixels_progressive(r._ctx, C.byref(args) if args is not None else None, C.c_void_p(p), n, C.c_void_p(a),
                                                C.c_void_p(s), C.c_void_p(c), first, None)

    for first in (1, 0):
        assert call(args=None, first=first) == RT_ERR_INVALID
        assert call(p=0, first=first) == RT_ERR_INVALID
        assert call(a=0, first=first) == RT_ERR_INVALID
        assert call(s=0, first=first) == RT_ERR_INVALID
        assert call(n=0, first=first) == RT_ERR_INVALID and call(n=-5, first=first) == RT_ERR_INVALID
        for bad in (rt.args(0, ny, ns, True), rt.args(nx, 0, ns, True), rt.args(nx, ny, 0, True),
                    rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_TILES, shard_rank=0, shard_count=2),
                    rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2),
                    rt.args(nx, ny, ns, True, seed_mode=7), rt.args(nx, ny, ns, True, precision=5)):
            assert call(args=bad, first=first) == RT_ERR_INVALID
        assert call(p=host_pix.ctypes.data, first=first) == RT_ERR_INVALID       # host memory would fault the GPU
        assert call(a=host_acc.ctypes.data, first=first) == RT_ERR_INVALID
        assert call(s=host_st.ctypes.data, first=first) == RT_ERR_INVALID
        assert call(c=host_cnt.ctypes.data, first=first) == RT_ERR_INVALID
    rt.build_octree(30, pkg.PREC_FP16)                                           # an octree for the other precision
    assert call() == RT_ERR_STATE
    rt.build_octree(30)
    assert call(args=rt.args(nx, ny, ns, True, precision=pkg.PREC_FP16)) == RT_ERR_STATE
    empty = pkg.RayTracer(0)
    try:
        assert call(r=empty) == RT_ERR_STATE                                     # no scene
        empty.create_world(488, 0.1)
        assert call(r=empty) == RT_ERR_STATE                                     # USE_OCTREE without an octree
    finally:
        empty.close()
    torch.cuda.synchronize()
    for t in (b.accum, b.state, b.counts):
        assert bool((t == 7).all())
    assert (host_acc == 7).all() and (host_st == 7).all() and (host_cnt == 7).all()
    fb = torch.zeros(npix * 3, dtype=torch.float32, device="cuda")
    L = rt.L
    for bad in (dict(a=0), dict(c=0), dict(f=0), dict(a=host_acc.ctypes.data), dict(c=host_cnt.ctypes.data), dict(f=host_acc.ctypes.data),
                dict(prec=2)):
        a, c, f = bad.get("a", b.accum.data_ptr()), bad.get("c", b.counts.data_ptr()), bad.get("f", fb.data_ptr())
        assert L.rt_finalize_counts(rt._ctx, C.c_void_p(a), C.c_void_p(c), C.c_void_p(f), npix, bad.get("prec", 0)) == RT_ERR_INVALID
    assert call() == 0 and call(c=0, first=0) == 0                               # counts are optional
    torch.cuda.synchronize()
    assert not bool((b.state == 7).all()) and bool((fb == 0).all()) and (host_acc == 7).all()


@gpu
@pytest.mark.parametrize("prec", [FP32, FP16], ids=["fp32", "fp16"])
def test_finalize_counts_uniform_counts_equal_rt_render(rt, pkg, prec):
    import torch
    rt.create_world(488, 0.1, prec)
    rt.build_octree(30, prec)
    nx, ny = 32, 16
    npix = nx * ny
    for ns in (1, 2, 3, 10, 64, 1000):
        b = Buffers(nx, ny)
        _frame_call(rt, rt.args(nx, ny, ns, True, precision=prec), b, True)
        b.counts.fill_(ns)
        got = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
        rt.finalize_counts(b.accum.data_ptr(), b.counts.data_ptr(), got.data_ptr(), npix, prec)
        ref = torch.empty_like(got)
        rt.render_device(rt.args(nx, ny, ns, True, precision=prec), ref.data_ptr())
        assert np.array_equal(_bits(_host(got)), _bits(_host(ref))), ns
        if prec == FP16:
            ex = torch.empty_like(got)
            rt.finalize_ex(b.accum.data_ptr(), ex.data_ptr(), npix * 3, ns, prec)
            assert np.array_equal(_bits(_host(got)), _bits(_host(ex))), ns
        rt.finalize_counts(b.accum.data_ptr(), b.counts.data_ptr(), b.accum.data_ptr(), npix, prec)    # in place
        assert np.array_equal(_bits(_host(b.accum)), _bits(_host(got))), ns
    b.counts.zero_()                                                              # count 0: zeros, whatever the sum
    b.accum.fill_(3.0)
    rt.finalize_counts(b.accum.data_ptr(), b.counts.data_ptr(), b.accum.data_ptr(), npix, prec)
    assert np.array_equal(_bits(_host(b.accum)), np.zeros(npix * 3, np.uint32))


@gpu
@pytest.mark.parametrize("ns", [1, 3, 10, 64, 1000])
def test_finalize_counts_fp16_every_half_value(rt, pkg, ns):
    """All 65 536 half bit patterns, widened to float, against col * real_t(1.0 / real_t(ns)) in half, sqrt in float, rounded to
    half (main.cu:111-115 under USE_FP16); every other pixel has count 0."""
    import torch
    acc16 = np.arange(1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    inv = np.float16(np.float32(1.0 / float(np.float16(ns))))
    with np.errstate(all="ignore"):
        want = np.float16(np.sqrt(np.float32(acc16 * inv))).astype(np.float32)
    acc = np.repeat(acc16.astype(np.float32), 2)                 # pixel k: (v[k/2], v[k/2], v[k/2]); odd pixels have count 0
    acc = np.repeat(acc, 3)
    counts = np.tile(np.array([ns, 0], np.uint32), 1 << 16)
    npix = len(counts)
    fb = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
    a, c = _dev(acc), _dev(counts)
    rt.finalize_counts(a.data_ptr(), c.data_ptr(), fb.data_ptr(), npix, pkg.PREC_FP16)
    got = _host(fb).reshape(-1, 2, 3)
    assert np.array_equal(_bits(got[:, 1]), np.zeros(((1 << 16), 3), np.uint32))
    got = got[:, 0]
    nan = np.isnan(want)
    assert np.isnan(got[nan]).all()
    assert np.array_equal(_bits(got[~nan]), _bits(np.repeat(want[~nan, None], 3, axis=1)))


@gpu
def test_integration_example(rt, pkg):
    """INTEGRATION.md's example: a 4-spp frame, 12 more samples on a window, then finalize_counts."""
    import torch
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    nx, ny = 120, 80
    accum = torch.empty(nx * ny * 3, dtype=torch.float32, device="cuda")
    state = torch.empty(nx * ny * 6, dtype=torch.int32, device="cuda")
    counts = torch.full((nx * ny,), 4, dtype=torch.int32, device="cuda")
    rt.render_progressive(rt.args(nx, ny, 4, True), accum.data_ptr(), state.data_ptr(), first=True)
    win = torch.from_numpy(pkg.window_pixels(nx, ny, 40, 88, 20, 52).view(np.int32)).cuda()
    rt.render_pixels_progressive(rt.args(nx, ny, 12, True), win.data_ptr(), win.numel(), accum.data_ptr(), state.data_ptr(),
                                 counts.data_ptr())
    fb = torch.empty_like(accum)
    rt.finalize_counts(accum.data_ptr(), counts.data_ptr(), fb.data_ptr(), nx * ny)
    got = _host(fb).reshape(ny, nx, 3)
    f4, _ = rt.render(nx, ny, 4)
    f16, _ = rt.render(nx, ny, 16)
    inside = np.zeros((ny, nx), bool)
    inside[20:52, 40:88] = True
    assert np.array_equal(_bits(got[inside]), _bits(f16[inside])) and np.array_equal(_bits(got[~inside]), _bits(f4[~inside]))


def _full_size(rt, pkg, nx, ny, pix, calls, ns, prec):
    """`calls` list-progressive calls of ns samples on the frame-indexed buffers, then finalize_counts -> fb[pix]."""
    import torch
    b = Buffers(nx, ny)
    p = _dev(pix)
    for k in range(calls):
        st = _list_call(rt, rt.args(nx, ny, ns, True, precision=prec), b, p, k == 0)
        assert st["paths"] == ns * len(np.unique(pix))
    fb = torch.empty(nx * ny * 3, dtype=torch.float32, device="cuda")
    rt.finalize_counts(b.accum.data_ptr(), b.counts.data_ptr(), fb.data_ptr(), nx * ny, prec)
    cnt = _host(b.counts, np.uint32)
    assert (cnt[pix] == calls * ns).all()
    return _host(fb).reshape(-1, 3)[pix]


@gpu
def test_config3_full_size_pixels_in_four_calls(rt, pkg, golden_dir):
    """BASELINE config 3 (3840x2160x64, 100 k spheres, SPHERES_PER_LEAF 300): the committed 1/16 x 1/16 subsample of the reference
    CUDA frame and the exact-tie pixels, as 4 list-progressive calls of 16 samples finalised from the counts."""
    nx, ny, n, spl = 3840, 2160, 100000, 300
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C3_3840x2160x64"]
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
    ties = json.load(open(os.path.join(golden_dir, "ref_cuda", "C3_tie_pixels.json")))
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).astype(np.uint32).reshape(-1)
    tp = np.array([j * nx + i for i, j in ties["pixels"]], np.uint32)
    got = _full_size(rt, pkg, nx, ny, np.concatenate([sub, tp]), 4, 16, FP32)
    assert np.array_equal(_bits(got[:len(sub)].reshape(gsub.shape)), _bits(gsub))
    want = np.array([[float.fromhex(h) for h in row] for row in ties["ref_gamma_f32_hex"]], np.float32)
    assert np.array_equal(_bits(got[len(sub):]), _bits(want))


@gpu
def test_config4_full_size_fp16_pixels_in_four_calls(rt, pkg, golden_dir):
    """BASELINE config 4 (USE_FP16, 4 spp): the committed 1/16 x 1/16 subsample of the reference's FP16 CUDA frame as 4
    list-progressive calls of 1 sample."""
    nx, ny, n, spl = 3840, 2160, 100000, 300
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C4_3840x2160x4"]
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"]))
    rt.create_world(n, 0.1, pkg.PREC_FP16)
    rt.build_octree(spl, pkg.PREC_FP16)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).astype(np.uint32).reshape(-1)
    got = _full_size(rt, pkg, nx, ny, sub, 4, 1, FP16)
    half = got.astype(np.float16)
    assert np.array_equal(half.astype(np.float32), got)
    assert np.array_equal(half.reshape(gsub.shape).view(np.uint16), gsub.view(np.uint16))
