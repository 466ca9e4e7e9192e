"""USE_FP16 frames in tile shards and progressive calls: rt_finalize_ex, k_render_h's sum and stream-state carry, and the
exchange of half sums between ranks.  The shard logic is proven on one GPU (every rank's shard rendered on cuda:0 into its own
buffer, summed with torch); only the NCCL and CLI cases need two GPUs."""
import ctypes as C
import json
import os
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RT_ERR_INVALID, RT_ERR_UNSUPPORTED = 10001, 10003

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


def _same(a, b):
    """Bit for bit, except that any NaN matches any NaN (a NaN's payload is not part of the image)."""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def _fp16_scene(rt, pkg, n, spl, octree):
    rt.create_world(n, 0.1, pkg.PREC_FP16)
    if octree:
        rt.build_octree(spl, pkg.PREC_FP16)


def _finalize_fp16(rt, pkg, acc, ns):
    import torch
    fb = torch.empty_like(acc)
    rt.finalize_ex(acc.data_ptr(), fb.data_ptr(), acc.numel(), ns, pkg.PREC_FP16)
    rt.synchronize()
    return fb.cpu().numpy()


# ---- CPU tier ----------------------------------------------------------------------------------------------------------------

def test_render_sharded_refuses_fp16_spp_shards_before_rendering():
    """render_sharded checks the combination before it touches the tracer or the frame (a stub that fails on any use)."""
    import __graft_entry__ as entry
    entry.load_package()
    from dd2360_raytracing_b200 import multigpu as mg

    class Untouchable:
        def __getattr__(self, name):
            raise AssertionError(f"render_sharded used {name} before refusing")

    frame = types.SimpleNamespace(world=2, rank=0, nx=8, ny=8)
    with pytest.raises(ValueError, match="tiles"):
        mg.render_sharded(Untouchable(), frame, 4, True, mode=mg.SHARD_SPP, precision=mg.PREC_FP16)


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("ns", [1, 2, 3, 4, 10, 64, 1000])
def test_finalize_ex_fp16_every_half_value(rt, pkg, ns):
    """All 65 536 half bit patterns, widened to float, against col * real_t(1.0 / real_t(ns)) in half, sqrt in float, rounded to
    half (main.cu:111-115 under USE_FP16)."""
    import torch
    acc16 = np.arange(1 << 16, dtype=np.uint32).astype(np.uint16).view(np.float16)
    inv = np.float16(np.float32(1.0 / float(np.float16(ns))))
    with np.errstate(all="ignore"):
        want = np.float16(np.sqrt(np.float32(acc16 * inv))).astype(np.float32)
    acc = torch.from_numpy(acc16.astype(np.float32)).cuda()
    got = _finalize_fp16(rt, pkg, acc, ns)
    nan = np.isnan(want)
    assert np.isnan(got[nan]).all()
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32))
    acc_in_place = acc.clone()                       # in place gives the same values
    rt.finalize_ex(acc_in_place.data_ptr(), acc_in_place.data_ptr(), acc.numel(), ns, pkg.PREC_FP16)
    rt.synchronize()
    assert _same(acc_in_place.cpu().numpy(), got)


@gpu
def test_finalize_ex_fp32_is_finalize_n(rt, pkg):
    import torch
    x = torch.from_numpy(np.random.default_rng(3).random(100003, dtype=np.float32) * 50).cuda()
    a, b = torch.empty_like(x), torch.empty_like(x)
    rt.finalize_n(x.data_ptr(), a.data_ptr(), x.numel(), 37)
    rt.finalize_ex(x.data_ptr(), b.data_ptr(), x.numel(), 37, pkg.PREC_FP32)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


PROGRESSIVE_CASES = [   # n, spl, octree, nx, ny, seed_mode, variant
    (488, 30, True, 96, 64, 0, 0),
    (488, 30, False, 40, 24, 0, 0),
    (8000, 30, True, 120, 80, 0, 0),
    (100000, 300, True, 192, 108, 0, 0),
    (8000, 30, True, 120, 80, 1, 0),          # upstream seeding: the stored states continue the skip-ahead streams
    (488, 30, True, 96, 64, 0, 30),           # 30, 32, 33: retired USE_FP16 variant numbers, which select the automatic kernel
    (488, 30, False, 40, 24, 0, 30),
    (8000, 30, True, 120, 80, 0, 32),
    (488, 30, False, 40, 24, 0, 32),
    (8000, 30, True, 120, 80, 0, 33),
]


@gpu
@pytest.mark.parametrize("n,spl,octree,nx,ny,seed_mode,variant", PROGRESSIVE_CASES)
def test_fp16_progressive_calls_equal_one_shot(rt, pkg, n, spl, octree, nx, ny, seed_mode, variant):
    """k calls of m samples == one k*m-sample render under USE_FP16: the half sums (resumed from the widened values), the stream
    states and the ray count, bit for bit; rt_finalize_ex of the sums is rt_render's FP16 frame."""
    import torch
    _fp16_scene(rt, pkg, n, spl, octree)
    total = 6
    kw = dict(seed_mode=seed_mode, variant=variant, precision=pkg.PREC_FP16)
    one = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    st1 = rt.render_accumulate(rt.args(nx, ny, total, octree, **kw), one.data_ptr())
    one = one.cpu().numpy()
    states = {}
    for chunks in ([1] * total, [2, 3, 1], [total]):
        acc = torch.full((ny, nx, 3), 7.0, dtype=torch.float32, device="cuda")        # garbage: the first call must overwrite it
        state = torch.zeros((ny * nx, 6), dtype=torch.int32, device="cuda")
        rays = 0
        for k, m in enumerate(chunks):
            st = rt.render_progressive(rt.args(nx, ny, m, octree, **kw), acc.data_ptr(), state.data_ptr(), first=(k == 0))
            rays += st["rays"]
        assert _same(acc.cpu().numpy(), one), chunks
        assert rays == st1["rays"], chunks
        states[tuple(chunks)] = state.cpu().numpy()
        frame = _finalize_fp16(rt, pkg, acc, total)
    first, *rest = states.values()
    assert all(np.array_equal(first, s) for s in rest)
    ref, _ = rt.render(nx, ny, total, use_octree=octree, **kw)
    assert _same(frame, ref)


SHARD_CASES = [   # n, spl, octree, nx, ny, variant, whether rank 1 renders its shard progressively
    (488, 30, True, 96, 64, 0, True),
    (488, 30, False, 40, 24, 0, False),
    (8000, 30, True, 120, 80, 0, False),
    (100000, 300, True, 192, 108, 0, True),
    (8000, 30, True, 120, 80, 32, False),     # 32: a retired variant number, which selects the automatic kernel
    (488, 30, False, 44, 26, 32, False),      # not a multiple of the 8x4 tile
]


@gpu
@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("n,spl,octree,nx,ny,variant,progressive", SHARD_CASES)
def test_fp16_tile_shards_add_up_to_the_one_gpu_frame(rt, pkg, G, n, spl, octree, nx, ny, variant, progressive):
    """Every rank's RT_SHARD_TILES shard rendered on one GPU into its own buffer: the buffers hold whole pixels' half sums and
    zeros, so their sum is the 1-GPU sum exactly, and rt_finalize_ex(FP16) of it is the one-shot FP16 frame.  Where marked, rank 1
    renders its shard progressively (2 + 3 samples)."""
    import torch
    _fp16_scene(rt, pkg, n, spl, octree)
    ns = 5
    kw = dict(variant=variant, precision=pkg.PREC_FP16)
    one = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    st1 = rt.render_accumulate(rt.args(nx, ny, ns, octree, **kw), one.data_ptr())
    bufs, rays = [], 0
    for g in range(G):
        buf = torch.full((ny, nx, 3), 7.0, dtype=torch.float32, device="cuda")
        sa = dict(shard_mode=pkg.SHARD_TILES, shard_rank=g, shard_count=G, **kw)
        if g == 1 and progressive:
            state = torch.zeros((ny * nx, 6), dtype=torch.int32, device="cuda")
            for k, m in enumerate((2, 3)):
                rays += rt.render_progressive(rt.args(nx, ny, m, octree, **sa), buf.data_ptr(), state.data_ptr(), first=(k == 0))["rays"]
        else:
            rays += rt.render_accumulate(rt.args(nx, ny, ns, octree, **sa), buf.data_ptr())["rays"]
        bufs.append(buf)
    acc = torch.stack(bufs).sum(0)
    assert _same(acc.cpu().numpy(), one.cpu().numpy()) and rays == st1["rays"]
    ref, _ = rt.render(nx, ny, ns, use_octree=octree, **kw)
    assert _same(_finalize_fp16(rt, pkg, acc, ns), ref)


@gpu
def test_config4_full_size_from_tiles_and_progressive_is_the_reference_fp16_frame(rt, pkg, golden_dir):
    """The C4 frame at 3840x2160x4 assembled from 3 tile shards on one GPU, and rendered progressively as 1 + 3 samples, both
    finalised by rt_finalize_ex(FP16): sha256 of the half framebuffer and of the PPM integers of the reference's FP16 CUDA build."""
    import sys
    import torch
    sys.path.insert(0, golden_dir)
    from digest_frame import digest
    man = json.load(open(os.path.join(golden_dir, "ref_cuda", "manifest_full.json")))["frames"]["C4_3840x2160x4"]
    nx, ny, ns, n, spl, G = 3840, 2160, 4, 100000, 300, 3
    try:
        _fp16_scene(rt, pkg, n, spl, True)
        acc = torch.zeros((ny, nx, 3), dtype=torch.float32, device="cuda")
        buf = torch.empty_like(acc)
        for g in range(G):
            rt.render_accumulate(rt.args(nx, ny, ns, True, shard_mode=pkg.SHARD_TILES, shard_rank=g, shard_count=G,
                                         precision=pkg.PREC_FP16), buf.data_ptr())
            acc += buf
        tiles = _finalize_fp16(rt, pkg, acc, ns)
        del acc
        prog = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
        state = torch.empty((ny * nx, 6), dtype=torch.int32, device="cuda")
        for k, m in enumerate((1, 3)):
            rt.render_progressive(rt.args(nx, ny, m, True, precision=pkg.PREC_FP16), prog.data_ptr(), state.data_ptr(), first=(k == 0))
        progressive = _finalize_fp16(rt, pkg, prog, ns)
        for frame in (tiles, progressive):
            d = digest(frame.astype(np.float16))          # half values widened to float: exact
            assert d["sha256_raw"] == man["sha256_raw"], d
            assert d["sha256_i32_ppm_order"] == man["sha256_i32_ppm_order"]
    finally:
        rt.create_world(488, 0.1)                          # leave the shared context in FP32
        rt.build_octree(30)


@gpu
def test_fp16_errors(rt, pkg):
    import torch
    from dd2360_raytracing_b200 import multigpu as mg
    L = pkg.load_library()
    _fp16_scene(rt, pkg, 488, 30, True)
    nx, ny = 40, 24
    buf = torch.full((ny, nx, 3), 7.0, dtype=torch.float32, device="cuda")
    a = rt.args(nx, ny, 4, True, shard_mode=pkg.SHARD_SPP, shard_rank=0, shard_count=2, precision=pkg.PREC_FP16)
    assert L.rt_render_accumulate(rt._ctx, C.byref(a), C.c_void_p(buf.data_ptr()), None) == RT_ERR_UNSUPPORTED
    assert b"tiles" in L.rt_last_error(rt._ctx)
    for prec, ns in ((7, 4), (-1, 4), (pkg.PREC_FP16, 0), (pkg.PREC_FP32, 0)):
        assert L.rt_finalize_ex(rt._ctx, C.c_void_p(buf.data_ptr()), C.c_void_p(buf.data_ptr()), buf.numel(), ns, prec) == RT_ERR_INVALID
    frame = mg.ShardedFrame(torch, torch.device("cuda", 0), nx, ny, 0, 2)
    frame.accum.fill_(7.0)
    with pytest.raises(ValueError, match="tiles"):
        mg.render_sharded(rt, frame, 4, True, mode=pkg.SHARD_SPP, precision=pkg.PREC_FP16)
    torch.cuda.synchronize()
    assert bool((frame.accum == 7.0).all()) and bool((buf == 7.0).all())       # nothing was rendered


# ---- two GPUs ----------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_fp16_c_abi_reduce_scatter_is_the_one_gpu_frame(pkg):
    """rt_comm_init_all + RT_SHARD_TILES per GPU + rt_reduce_scatter + rt_finalize_ex(FP16) through the C ABI, one process driving
    two GPUs: the 1-GPU FP16 frame bit for bit."""
    import torch
    L = pkg.load_library()
    G = 2
    nx, ny, ns, n, spl = 240, 160, 6, 8000, 30
    rts = [pkg.RayTracer(g) for g in range(G)]
    try:
        for r in rts:
            _fp16_scene(r, pkg, n, spl, True)
        ref, _ = rts[0].render(nx, ny, ns, precision=pkg.PREC_FP16)
        arr = (C.c_void_p * G)(*[r._ctx for r in rts])
        assert L.rt_comm_init_all(arr, G) == 0, L.rt_last_error(rts[0]._ctx)
        total = nx * ny * 3
        S = (total + G - 1) // G
        acc = [torch.zeros(S * G, dtype=torch.float32, device=f"cuda:{g}") for g in range(G)]
        sl = [torch.empty(S, dtype=torch.float32, device=f"cuda:{g}") for g in range(G)]
        for g, r in enumerate(rts):
            r.render_accumulate(r.args(nx, ny, ns, True, shard_mode=pkg.SHARD_TILES, shard_rank=g, shard_count=G, precision=pkg.PREC_FP16),
                                acc[g].data_ptr())
        assert L.rt_group_start() == 0
        for g, r in enumerate(rts):
            assert L.rt_reduce_scatter(r._ctx, C.c_void_p(acc[g].data_ptr()), C.c_void_p(sl[g].data_ptr()), S) == 0
        assert L.rt_group_end() == 0
        for g, r in enumerate(rts):
            r.finalize_ex(sl[g].data_ptr(), sl[g].data_ptr(), S, ns, pkg.PREC_FP16)
            r.synchronize()
        frame = torch.cat([s.cpu() for s in sl])[:total].view(ny, nx, 3).numpy()
        assert _same(frame, ref)
    finally:
        for r in rts:
            L.rt_comm_destroy(r._ctx)
            r.close()


_WORKER = r'''
import json, os, sys
import numpy as np
import torch
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
import __graft_entry__ as entry
pkg = entry.load_package()
from dd2360_raytracing_b200 import multigpu as mg
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
nx, ny, ns = 240, 160, 6
rt = pkg.RayTracer(rank)
rt.set_stream(torch.cuda.current_stream().cuda_stream)
rt.create_world(8000, 0.1, pkg.PREC_FP16)
rt.build_octree(30, pkg.PREC_FP16)
frame = mg.ShardedFrame(torch, torch.device("cuda", rank), nx, ny, rank, world)
mg.render_sharded(rt, frame, ns, True, mode=pkg.SHARD_TILES, dist=dist, precision=pkg.PREC_FP16)
slices = [torch.empty_like(frame.slice) for _ in range(world)]
dist.all_gather(slices, frame.slice)
torch.cuda.synchronize()
if rank == 0:
    got = torch.cat(slices)[: frame.total].view(ny, nx, 3).cpu().numpy()
    ref, _ = rt.render(nx, ny, ns, precision=pkg.PREC_FP16)
    same = ((got.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(got) & np.isnan(ref))).all()
    print(json.dumps({"identical": bool(same)}))
dist.barrier()
dist.destroy_process_group()
rt.close()
'''


@gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_fp16_torch_distributed_frame_is_the_one_gpu_frame(tmp_path):
    """multigpu.render_sharded(precision=PREC_FP16) on two torch.distributed ranks (NCCL reduce-scatter, per-rank rt_finalize_ex)."""
    import subprocess
    import sys
    worker = tmp_path / "fp16_worker.py"
    worker.write_text(_WORKER)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29579", str(worker), ROOT]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["identical"] is True


@gpu
@pytest.mark.skipif(_gpu_count() < 2, reason="needs two GPUs")
def test_fp16_cli_on_two_gpus_writes_the_one_gpu_file(pkg, tmp_path):
    """`RT_GPUS=2 RT_USE_FP16=1 ./RayTracing 3` shards by tiles and writes the 1-GPU output.ppm byte for byte; RT_SHARD=spp is refused."""
    import subprocess
    exe = os.path.join(os.path.dirname(pkg.LIB_PATH), "RayTracing")
    env = dict(os.environ, RT_NUM_SPHERES="8000", RT_SPHERES_PER_LEAF="30", RT_NX="400", RT_NY="240", RT_NS="4", RT_USE_FP16="1")
    files = {}
    for gpus in ("1", "2"):
        d = tmp_path / f"g{gpus}"
        d.mkdir()
        subprocess.run([exe, "3"], cwd=d, env=dict(env, RT_GPUS=gpus), capture_output=True, check=True, timeout=600)
        files[gpus] = (d / "output.ppm").read_bytes()
    assert files["1"].startswith(b"P3\n400 240\n255\n") and files["2"] == files["1"]
    r = subprocess.run([exe, "3"], cwd=tmp_path, env=dict(env, RT_GPUS="2", RT_SHARD="spp"), capture_output=True, timeout=600)
    assert r.returncode != 0 and b"tiles" in r.stderr
