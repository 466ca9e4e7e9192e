"""rt_render_adaptive: adaptive sampling over the frame queue's 8x4 tiles.

Every pixel of an adaptive frame is held, bit for bit, to one-shot renders at its own count (sum and stream state to the one-shot
progressive render, the frame to rt_render(ns = count)) on every kernel path, and the counts, the per-pixel errors and the rounds
to a numpy model of the decision procedure built from one-shot sums at every level.  Frames are 203x117 unless stated, so the
edge tiles are partial."""
import ctypes as C
import json
import math
import os

import numpy as np
import pytest

from test_adaptive_host import metric_model
from test_gpu_pixel_progressive import CASES, Buffers, _bits, _dev, _host, _oneshot

RT_ERR_INVALID, RT_ERR_STATE = 10001, 10002
NX, NY = 203, 117

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


def _gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _scene(rt, n, spl, prec):
    rt.create_world(n, 0.1, prec)
    if spl is not None:
        rt.build_octree(spl, prec)


def _adaptive(rt, nx, ny, max_spp, min_spp, thr, octree, kw):
    """One rt_render_adaptive call on fresh buffers -> (Buffers, fb[npix, 3], err[npix], stats)."""
    import torch
    b = Buffers(nx, ny)
    fb = torch.empty(nx * ny * 3, dtype=torch.float32, device="cuda")
    err = torch.empty(nx * ny, dtype=torch.float32, device="cuda")
    st = rt.render_adaptive_device(rt.args(nx, ny, max_spp, octree, **kw), min_spp, thr, b.accum.data_ptr(), b.state.data_ptr(),
                                   b.counts.data_ptr(), fb.data_ptr(), err.data_ptr())
    return b, _host(fb).reshape(-1, 3), _host(err), st


def _levels(min_spp, max_spp):
    lv, c = [min_spp // 2, min_spp], min_spp
    while c < max_spp:
        c += min(c, max_spp - c)
        lv.append(c)
    return lv


class OneShots:
    """One-shot (sums, states, rt_render frame) of a scene at any sample count, computed once each."""

    def __init__(self, rt, nx, ny, octree, kw):
        self.rt, self.nx, self.ny, self.octree, self.kw, self.cache = rt, nx, ny, octree, kw, {}

    def __call__(self, S):
        if S not in self.cache:
            self.cache[S] = _oneshot(self.rt, self.nx, self.ny, int(S), self.octree, self.kw)
        return self.cache[S]


def _tile_of(nx, ny):
    j, i = np.divmod(np.arange(nx * ny), nx)
    return (j // 4) * ((nx + 7) // 8) + i // 8


def model(pkg, shots, nx, ny, min_spp, max_spp, thr):
    """The decision procedure restated: -> (counts[npix], err[npix], [list of round r])."""
    npix, tiles = nx * ny, ((nx + 7) // 8) * ((ny + 3) // 4)
    tile_of = _tile_of(nx, ny)
    counts = np.full(npix, min_spp, np.uint32)
    err = np.zeros(npix, np.float32)
    done = np.zeros(tiles, bool)
    a, c, rounds = min_spp // 2, min_spp, []
    thr = np.float32(thr)
    while True:
        act = ~done[tile_of]
        A, X = shots(a)[0][act], shots(c)[0][act]
        e = metric_model(A, np.full(len(A), a, np.uint32), X, np.full(len(A), c, np.uint32))
        err[act] = e
        E = np.zeros(tiles, np.float32)
        np.maximum.at(E, tile_of[act], np.where(np.isnan(e), np.float32(np.inf), e))
        refine = ~done & (c < max_spp) & ~(E <= thr)
        done |= ~refine
        if not refine.any():
            break
        # tiles row-major, each tile's in-frame pixels row by row
        lst = np.array([j * nx + i for t in np.nonzero(refine)[0]
                        for j in range((t // ((nx + 7) // 8)) * 4, min((t // ((nx + 7) // 8)) * 4 + 4, ny))
                        for i in range((t % ((nx + 7) // 8)) * 8, min((t % ((nx + 7) // 8)) * 8 + 8, nx))], np.uint32)
        wp = pkg.window_pixels(nx, ny, 0, nx, 0, ny)
        assert np.array_equal(lst, wp[refine[tile_of[wp]]])
        more = min(c, max_spp - c)
        counts[refine[tile_of]] = c + more
        rounds.append(lst)
        a, c = c, c + more
    return counts, err, rounds


def _tile_errors(shots, nx, ny, a, c):
    tile_of = _tile_of(nx, ny)
    e = metric_model(shots(a)[0], np.full(nx * ny, a, np.uint32), shots(c)[0], np.full(nx * ny, c, np.uint32))
    E = np.zeros(tile_of.max() + 1, np.float32)
    np.maximum.at(E, tile_of, np.where(np.isnan(e), np.float32(np.inf), e))
    return E


def _pick_threshold(pkg, shots, nx, ny, min_spp, max_spp):
    """A threshold (a quantile of the first round's tile errors) at which the model gives at least three distinct counts."""
    E = _tile_errors(shots, nx, ny, min_spp // 2, min_spp)
    for q in (0.5, 0.35, 0.65, 0.2, 0.8, 0.9):
        thr = float(np.quantile(E[np.isfinite(E)], q))
        counts, _, _ = model(pkg, shots, nx, ny, min_spp, max_spp, thr)
        if len(np.unique(counts)) >= 3:
            return thr
    raise AssertionError("no threshold gives three distinct counts")


def _same_err(got, want):
    nan = np.isnan(want)
    return bool((np.isnan(got) == nan).all() and np.array_equal(_bits(got[~nan]), _bits(want[~nan])))


def _check_exact(b, fb, shots, what):
    """Every pixel's sum and state equal the one-shot progressive render at its count, and fb equals rt_render(ns = count)."""
    acc, st, cnt = b.host()
    for S in np.unique(cnt):
        ref_acc, ref_st, ref_fb = shots(int(S))
        m = cnt == S
        for name, got, want in (("accum", _bits(acc[m]), _bits(ref_acc[m])), ("state", st[m], ref_st[m]), ("fb", _bits(fb[m]), _bits(ref_fb[m]))):
            bad = np.nonzero((got != want).any(axis=1))[0]
            assert len(bad) == 0, (what, name, int(S), int(np.nonzero(m)[0][bad[0]]))


def _check_model(pkg, b, err, st, shots, nx, ny, min_spp, max_spp, thr, what):
    counts, merr, rounds = model(pkg, shots, nx, ny, min_spp, max_spp, thr)
    cnt = b.host()[2]
    assert np.array_equal(cnt, counts), what
    assert _same_err(err, merr), what
    assert st["rounds"] == len(rounds) and st["round_pixels"] == [len(r) for r in rounds], (what, st)
    tile_of = _tile_of(nx, ny)
    first = np.zeros(tile_of.max() + 1, np.uint32)
    first[tile_of[::-1]] = cnt[::-1]
    assert np.array_equal(cnt, first[tile_of]), "counts differ inside a tile"
    return counts


# ---- 1, 2: every kernel path against one-shot renders, and the decision procedure against the model --------------------------

@gpu
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_adaptive_frames_equal_one_shot_renders(rt, pkg, case):
    name, n, spl, prec, variant, kernel = case
    octree = spl is not None
    _scene(rt, n, spl, prec)
    min_spp, max_spp = 2, 16
    for seed in (pkg.SEED_HEAD, pkg.SEED_UPSTREAM):
        kw = dict(seed_mode=seed, precision=prec, variant=variant)
        shots = OneShots(rt, NX, NY, octree, kw)
        thr = _pick_threshold(pkg, shots, NX, NY, min_spp, max_spp)
        b, fb, err, st = _adaptive(rt, NX, NY, max_spp, min_spp, thr, octree, kw)
        assert st["kernel"].startswith(kernel), st["kernel"]
        counts = _check_model(pkg, b, err, st, shots, NX, NY, min_spp, max_spp, thr, (name, seed))
        assert len(np.unique(counts)) >= 3
        _check_exact(b, fb, shots, (name, seed))
        assert st["paths"] == int(counts.astype(np.int64).sum())


# ---- 3: bounds ----------------------------------------------------------------------------------------------------------------

@gpu
def test_bounds(rt, pkg):
    _scene(rt, 488, 30, 0)
    kw = {}
    shots = OneShots(rt, NX, NY, True, kw)
    npix = NX * NY
    # threshold +inf: a uniform min_spp frame, no rounds
    b, fb, err, st = _adaptive(rt, NX, NY, 64, 4, float("inf"), True, kw)
    assert st["rounds"] == 0 and (b.host()[2] == 4).all()
    assert np.array_equal(_bits(fb), _bits(shots(4)[2]))
    _check_model(pkg, b, err, st, shots, NX, NY, 4, 64, float("inf"), "inf")
    # threshold 0: every tile whose error is not 0 goes on to max_spp
    b, fb, err, st = _adaptive(rt, NX, NY, 16, 2, 0.0, True, kw)
    cnt = _check_model(pkg, b, err, st, shots, NX, NY, 2, 16, 0.0, "zero")
    tile_of = _tile_of(NX, NY)
    E = np.zeros(tile_of.max() + 1, np.float32)
    np.maximum.at(E, tile_of, np.where(np.isnan(err), np.float32(np.inf), err))
    assert ((cnt == 16) | (E[tile_of] == 0)).all() and (cnt == 16).mean() > 0.5
    _check_exact(b, fb, shots, "zero")
    # max_spp == min_spp: no rounds, but every pixel's estimate from its two halves
    b, fb, err, st = _adaptive(rt, NX, NY, 6, 6, 0.0, True, kw)
    assert st["rounds"] == 0 and (b.host()[2] == 6).all()
    _check_model(pkg, b, err, st, shots, NX, NY, 6, 6, 0.0, "min == max")
    assert np.array_equal(_bits(fb), _bits(shots(6)[2]))
    # max_spp not min * 2^k: the last round is capped (2, 4, 8, then 4 more to 12)
    b, fb, err, st = _adaptive(rt, NX, NY, 12, 2, 0.0, True, kw)
    cnt = _check_model(pkg, b, err, st, shots, NX, NY, 2, 12, 0.0, "capped")
    assert st["rounds"] == 3 and cnt.max() == 12 and _levels(2, 12) == [1, 2, 4, 8, 12]
    _check_exact(b, fb, shots, "capped")
    assert st["paths"] == int(cnt.astype(np.int64).sum()) and npix * 2 <= st["paths"] <= npix * 12


# ---- 4, 5: determinism, continuation, stats ---------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("prec", [0, 1], ids=["fp32", "fp16"])
def test_determinism_continuation_and_stats(rt, pkg, prec):
    import torch
    _scene(rt, 488, 30, prec)
    kw = dict(precision=prec, seed_mode=pkg.SEED_UPSTREAM)
    shots = OneShots(rt, NX, NY, True, kw)
    thr = _pick_threshold(pkg, shots, NX, NY, 4, 32)
    runs = [_adaptive(rt, NX, NY, 32, 4, thr, True, kw) for _ in range(2)]
    (b1, fb1, err1, st1), (b2, fb2, err2, st2) = runs
    for x, y in zip(b1.host() + (fb1, err1), b2.host() + (fb2, err2)):
        assert np.ascontiguousarray(x).tobytes() == np.ascontiguousarray(y).tobytes()
    assert {k: v for k, v in st1.items() if k != "kernel_ms"} == {k: v for k, v in st2.items() if k != "kernel_ms"}
    # stats: paths = sum of the counts; rays = the rays of each count group rendered as a pixel list at its count
    cnt = b1.host()[2]
    assert st1["paths"] == int(cnt.astype(np.int64).sum())
    rays = 0
    for S in np.unique(cnt):
        _, s = rt.render_pixels(NX, NY, int(S), np.nonzero(cnt == S)[0].astype(np.uint32), True, **kw)
        rays += s["rays"]
    assert st1["rays"] == rays and st1["kernel_ms"] > 0 and st1["rounds"] >= 2
    # continuation: 3 more samples on a window through rt_render_pixels_progressive end at the one-shot render of count + 3
    win = pkg.window_pixels(NX, NY, 37, 150, 10, 90)
    rt.render_pixels_progressive(rt.args(NX, NY, 3, True, **kw), _dev(win).data_ptr(), len(win), b1.accum.data_ptr(), b1.state.data_ptr(),
                                 b1.counts.data_ptr())
    acc, st, cnt2 = b1.host()
    assert np.array_equal(cnt2[win], cnt[win] + 3)
    for S in np.unique(cnt2[win]):
        ref_acc, ref_st, _ = shots(int(S))
        m = win[cnt2[win] == S]
        assert np.array_equal(_bits(acc[m]), _bits(ref_acc[m])) and np.array_equal(st[m], ref_st[m]), int(S)
    torch.cuda.synchronize()


# ---- 6: errors ----------------------------------------------------------------------------------------------------------------

@gpu
def test_errors_write_nothing(rt, pkg):
    import torch
    _scene(rt, 488, 30, 0)
    nx, ny = 40, 24
    npix = nx * ny
    b = Buffers(nx, ny)
    fb = torch.empty(npix * 3, dtype=torch.float32, device="cuda")
    err = torch.empty(npix, dtype=torch.float32, device="cuda")
    for t in (b.accum, fb, err):
        t.view(torch.int32).fill_(0x7FA5A5A5)
    b.state.fill_(-0x5A5A5A5B)
    b.counts.fill_(0x13579BD)
    host = np.full(npix * 6, 7, np.uint32)
    good = rt.args(nx, ny, 16, True)

    def call(r=rt, args=good, min_spp=2, thr=0.01, params=True, a=None, s=None, c=None, f=None, e=None):
        p = pkg.AdaptiveParams(min_spp, thr)
        ptr = lambda v, d: C.c_void_p(d.data_ptr() if v is None else v)
        return r.L.rt_render_adaptive(r._ctx, C.byref(args) if args is not None else None, C.byref(p) if params else None,
                                      ptr(a, b.accum), ptr(s, b.state), ptr(c, b.counts), ptr(f, fb), ptr(e, err), None)

    before = [t.clone() for t in (b.accum, b.state, b.counts, fb, err)]
    assert call(args=None) == RT_ERR_INVALID and call(params=False) == RT_ERR_INVALID
    for k in ("a", "s", "c", "f"):
        assert call(**{k: 0}) == RT_ERR_INVALID, k
        assert call(**{k: host.ctypes.data}) == RT_ERR_INVALID, k          # host memory would fault the GPU
    assert call(e=host.ctypes.data) == RT_ERR_INVALID
    for m in (0, 1, 3, -2, 7):
        assert call(min_spp=m) == RT_ERR_INVALID, m
    for ns in (1, 0, -4, 65537):
        assert call(args=rt.args(nx, ny, ns, True)) == RT_ERR_INVALID, ns
    assert call(min_spp=18) == RT_ERR_INVALID                                  # max_spp < min_spp
    for thr in (float("nan"), -1e-9, -1.0, float("-inf")):
        assert call(thr=thr) == RT_ERR_INVALID, thr
    for bad in (rt.args(0, ny, 16, True), rt.args(nx, 0, 16, True),
                rt.args(nx, ny, 16, True, shard_mode=pkg.SHARD_TILES, shard_rank=0, shard_count=2),
                rt.args(nx, ny, 16, True, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2),
                rt.args(nx, ny, 16, True, seed_mode=7), rt.args(nx, ny, 16, True, precision=5)):
        assert call(args=bad) == RT_ERR_INVALID
    rt.build_octree(30, pkg.PREC_FP16)                                          # an octree for the other precision
    assert call() == RT_ERR_STATE
    rt.build_octree(30)
    assert call(args=rt.args(nx, ny, 16, True, precision=pkg.PREC_FP16)) == RT_ERR_STATE
    empty = pkg.RayTracer(0)
    try:
        assert call(r=empty) == RT_ERR_STATE                                   # no scene
        empty.create_world(488, 0.1)
        assert call(r=empty) == RT_ERR_STATE                                   # USE_OCTREE without an octree
    finally:
        empty.close()
    torch.cuda.synchronize()
    for x, y in zip(before, (b.accum, b.state, b.counts, fb, err)):
        assert bool((x.view(torch.int32) == y.view(torch.int32)).all())
    assert (host == 7).all()
    assert call() == 0 and call(e=0) == 0 and call(thr=0.0) == 0 and call(thr=float("inf")) == 0     # err is optional
    torch.cuda.synchronize()


# ---- 7: quality ---------------------------------------------------------------------------------------------------------------

def _psnr(fb, ref):
    mse = float(np.mean((fb.astype(np.float64) - ref.astype(np.float64)) ** 2))
    return 10.0 * math.log10(1.0 / mse), mse


QUALITY_THRESHOLD = 2.0 / 255


@gpu
def test_quality_beats_uniform_at_the_same_cost(rt, pkg):
    """488 spheres in an octree at 400x225, min 8, max 256, threshold 2/255, against the uniform 1024-spp frame: adaptive's PSNR is
    above that of a uniform frame of U = ceil(paths / npix) samples.  Measured on a B200 (everything is seeded, so deterministic):
    adaptive 48.42 dB at 148.5 spp on average (rounds of 62 048, 61 920, 60 480, 53 664 and 45 248 pixels), uniform-149 45.74 dB:
    a margin of 2.68 dB."""
    _scene(rt, 488, 30, 0)
    nx, ny = 400, 225
    ref, _ = rt.render(nx, ny, 1024)
    fb, counts, err, st = rt.render_adaptive(nx, ny, 256, 8, QUALITY_THRESHOLD)
    U = -(-st["paths"] // (nx * ny))
    uni, _ = rt.render(nx, ny, U)
    p_ad, _ = _psnr(fb, ref)
    p_un, _ = _psnr(uni, ref)
    print(f"adaptive {p_ad:.3f} dB ({st['paths'] / (nx * ny):.2f} spp, rounds {st['round_pixels']}), uniform-{U} {p_un:.3f} dB")
    assert counts.min() >= 8 and counts.max() <= 256 and len(np.unique(counts)) >= 3
    assert p_ad > p_un


# ---- 8: full size -------------------------------------------------------------------------------------------------------------

@gpu
def test_config3_full_size_pixels_at_64_equal_the_golden(rt, pkg, golden_dir):
    """BASELINE config 3 (3840x2160, 100 k spheres, SPHERES_PER_LEAF 300) with max_spp 64: every pixel of the committed 1/16 x 1/16
    subsample of the reference CUDA frame that ends at 64 samples equals it, and so does each exact-tie pixel that ends at 64."""
    nx, ny, n, spl = 3840, 2160, 100000, 300
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C3_3840x2160x64"]
    gsub = np.load(os.path.join(golden_dir, "ref_cuda", man["subsample"])).reshape(-1, 3)
    ties = json.load(open(os.path.join(golden_dir, "ref_cuda", "C3_tie_pixels.json")))
    _scene(rt, n, spl, 0)
    fb, counts, err, st = rt.render_adaptive(nx, ny, 64, 8, 1.0 / 255)
    fb, counts = fb.reshape(-1, 3), counts.reshape(-1)
    jj, ii = np.meshgrid(np.arange(0, ny, 16), np.arange(0, nx, 16), indexing="ij")
    sub = (jj * nx + ii).reshape(-1)
    at64 = counts[sub] == 64
    assert at64.sum() > 0 and (counts[sub][~at64] < 64).all()
    assert np.array_equal(_bits(fb[sub[at64]]), _bits(gsub[at64]))
    want = np.array([[float.fromhex(h) for h in row] for row in ties["ref_gamma_f32_hex"]], np.float32)
    tp = np.array([j * nx + i for i, j in ties["pixels"]])
    m = counts[tp] == 64
    assert np.array_equal(_bits(fb[tp[m]]), _bits(want[m]))


# ---- 9: CLI -------------------------------------------------------------------------------------------------------------------

@gpu
def test_cli_writes_the_adaptive_frame(rt, pkg, tmp_path):
    """`RT_ADAPTIVE=<threshold>:<min> ./RayTracing 3` writes output.ppm byte for byte as rt_format_ppm of render_adaptive's frame."""
    import subprocess
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "RayTracing")
    env = dict(os.environ, RT_NUM_SPHERES="488", RT_SPHERES_PER_LEAF="30", RT_NX="320", RT_NY="180", RT_NS="32",
               RT_ADAPTIVE="0.01:4", RT_VERBOSE="1")
    r = subprocess.run([exe, "3"], cwd=tmp_path, env=env, capture_output=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert b"rounds" in r.stderr and b"mean" in r.stderr
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    fb, counts, _, _ = rt.render_adaptive(320, 180, 32, 4, 0.01)
    assert len(np.unique(counts)) >= 2
    assert (tmp_path / "output.ppm").read_bytes() == pkg.format_ppm(fb)


@gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_cli_refuses_adaptive_on_two_gpus(pkg, tmp_path):
    import subprocess
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "RayTracing")
    env = dict(os.environ, RT_NUM_SPHERES="488", RT_NX="64", RT_NY="32", RT_NS="8", RT_ADAPTIVE="0.01", RT_GPUS="2")
    r = subprocess.run([exe, "3"], cwd=tmp_path, env=env, capture_output=True, timeout=600)
    assert r.returncode != 0 and b"one GPU" in r.stderr
