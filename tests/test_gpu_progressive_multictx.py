"""GPU tier (-m gpu): progressive rendering with state carry (main.cu:119-142), per-context cameras, kernel reporting,
and the multi-GPU C ABI (NCCL; needs >= 2 GPUs, skipped otherwise)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


@pytest.mark.parametrize("n,spl,octree,nx,ny,seed_mode,variant", [
    (488, 30, True, 96, 64, 0, 0),
    (488, 30, False, 40, 24, 0, 0),
    (8000, 30, True, 120, 80, 0, 1),        # the pixel-per-lane kernel
    (8000, 30, True, 120, 80, 1, 0),        # upstream seeding: the stored states continue the skip-ahead streams
    (100000, 300, True, 192, 108, 0, 11),   # 11 (the retired pooled kernel) selects the automatic choice: the cooperative kernel
])
def test_progressive_calls_equal_one_shot(rt, pkg, n, spl, octree, nx, ny, seed_mode, variant):
    """k calls of m samples == one k*m-sample render: linear sums, final frame and stream states, bit for bit —
    what render_progressive's stored rand_state (main.cu:136) and fb += col (main.cu:141) give the reference."""
    import torch
    rt.create_world(n, 0.1)
    if octree:
        rt.build_octree(spl)
    total = 6
    one = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    st1 = rt.render_accumulate(rt.args(nx, ny, total, octree, seed_mode=seed_mode, variant=variant), one.data_ptr())
    for chunks in ([1] * total, [2, 3, 1], [total]):
        acc = torch.full((ny, nx, 3), 7.0, dtype=torch.float32, device="cuda")        # garbage: the first call must overwrite it
        state = torch.zeros((ny * nx, 6), dtype=torch.int32, device="cuda")
        rays = 0
        for k, m in enumerate(chunks):
            st = rt.render_progressive(rt.args(nx, ny, m, octree, seed_mode=seed_mode, variant=variant), acc.data_ptr(), state.data_ptr(), first=(k == 0))
            rays += st["rays"]
        assert torch.equal(acc.view(torch.int32), one.view(torch.int32)), chunks
        assert rays == st1["rays"]
    # a dump in the middle is a valid frame of the samples so far
    fb = torch.empty_like(one)
    rt.finalize(acc.data_ptr(), fb.data_ptr(), nx, ny, total)
    ref, _ = rt.render(nx, ny, total, use_octree=octree, seed_mode=seed_mode, variant=variant)
    assert np.array_equal(fb.cpu().numpy().view(np.uint32), ref.view(np.uint32))


def test_two_contexts_keep_their_own_cameras(pkg, O):
    """The camera is per-context state (it used to live in one __constant__ symbol per library): two live contexts on one
    GPU with different frame sizes and a custom camera render what each was told to, in any order."""
    a, b = pkg.RayTracer(0), pkg.RayTracer(0)
    try:
        for r in (a, b):
            r.create_world(488, 0.1)
            r.build_octree(30)
        desc = pkg.CameraDesc((C.c_float * 3)(3, 4, 10), (C.c_float * 3)(0, 0.5, 0), (C.c_float * 3)(0, 1, 0), 40.0, 1.25, 0.0, 8.0)
        fa0, _ = a.render(96, 64, 2)
        b.set_camera(80, 64, desc)
        fb0, _ = b.render(80, 64, 2)
        fa1, _ = a.render(96, 64, 2)             # b's camera upload must not have leaked into a
        fb1, _ = b.render(80, 64, 2)
        assert np.array_equal(fa0.view(np.uint32), fa1.view(np.uint32)) and np.array_equal(fb0.view(np.uint32), fb1.view(np.uint32))
        sph, _ = O.create_world(488)
        blob, _ = O.build_octree(sph, 30)
        ref, _, _ = O.render(sph, O.camera(96, 64, O.ARITH_DEVICE), O.make_params(96, 64, 2, True, 30, O.ARITH_DEVICE), blob)
        assert np.array_equal(fa1.view(np.uint32), ref.view(np.uint32))
        # a custom description survives a change of frame size (it is not silently replaced by the main.cu camera)
        cam_before = b.camera().copy()
        b.render(40, 32, 1)
        assert np.array_equal(b.camera(), cam_before)
    finally:
        a.close()
        b.close()


def test_stats_name_the_kernel_that_ran(rt, pkg):
    rt.create_world(488, 0.1)
    rt.build_octree(30)
    _, s = rt.render(64, 40, 1, use_octree=True, variant=1)
    assert s["kernel"].startswith("k_render<octree>")
    _, s = rt.render(64, 40, 1, use_octree=True, variant=40)
    assert s["kernel"].startswith("k_render_coop")
    _, s = rt.render(64, 40, 1, use_octree=True, variant=11)      # a retired variant number: the automatic choice for 488 spheres
    assert s["kernel"].startswith("k_render<octree>")


def test_cooperative_and_per_lane_kernels_agree(rt):
    """k_render_coop (variant 40) against k_render (variant 1) on scenes of every size class, flat list through the grid included."""
    import torch
    for n, spl, octree, nx, ny, ns in [(488, 30, True, 240, 160, 4), (488, 30, False, 240, 160, 2), (8000, 30, True, 240, 160, 3),
                                       (20000, 30, True, 160, 96, 2), (100000, 300, True, 480, 270, 2), (1000000, 3000, True, 192, 108, 1)]:
        rt.create_world(n, 0.1)
        if octree:
            rt.build_octree(spl)
        out = []
        for v in (1, 40):
            fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
            st = rt.render_device(rt.args(nx, ny, ns, octree, variant=v), fb.data_ptr())
            out.append((fb, st["rays"]))
        same = float((out[0][0] == out[1][0]).all(dim=2).float().mean())
        assert same >= 1 - 1e-5 and abs(out[0][1] - out[1][1]) <= 4, (n, same, out[0][1], out[1][1])


def test_voxel_shape_is_only_a_speed_knob(pkg, monkeypatch):
    """choose_grid's flat voxels (slab-shaped scenes from 40 k spheres; RT_GRID_SHAPE is read when a context is created): cubes, the
    default and very flat voxels render the same frame, through the cooperative and the per-lane kernel."""
    import torch
    nx, ny, ns = 192, 108, 2
    frames, grids = [], []
    for shape in ("1:1", None, "3:0.5"):
        if shape is None:
            monkeypatch.delenv("RT_GRID_SHAPE", raising=False)
        else:
            monkeypatch.setenv("RT_GRID_SHAPE", shape)
        r = pkg.RayTracer(0)
        try:
            r.create_world(100000, 0.1)
            st = r.build_octree(300)
            grids.append((st["fine_voxels"], st["fine_refs"]))
            for variant in (0, 1):
                fb = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
                r.render_device(r.args(nx, ny, ns, True, variant=variant), fb.data_ptr())
                frames.append(fb.cpu().numpy())
        finally:
            r.close()
    assert len(set(grids)) == 3, grids                       # the knob did change the grid
    for f in frames[1:]:
        assert np.array_equal(f.view(np.uint32), frames[0].view(np.uint32))


def _multi_gpu_count():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_multi_gpu_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("mode", ["tiles", "spp"])
def test_c_abi_multi_gpu_reduce(pkg, mode):
    """rt_comm_init_all + rt_render_accumulate per GPU + rt_reduce / rt_reduce_scatter (NCCL) through the C ABI, one process
    driving two GPUs: tile shards reproduce the 1-GPU frame bit for bit; spp shards give a frame of the same radiance."""
    import torch
    L = pkg.load_library()
    G = 2
    nx, ny, ns, n, spl = 240, 160, 8, 8000, 30
    rts = [pkg.RayTracer(g) for g in range(G)]
    try:
        for r in rts:
            r.create_world(n, 0.1)
            r.build_octree(spl)
        ref, _ = rts[0].render(nx, ny, ns)
        arr = (C.c_void_p * G)(*[r._ctx for r in rts])
        assert L.rt_comm_init_all(arr, G) == 0, L.rt_last_error(rts[0]._ctx)
        total = nx * ny * 3
        S = (total + G - 1) // G
        acc = [torch.zeros(S * G, dtype=torch.float32, device=f"cuda:{g}") for g in range(G)]
        sl = [torch.empty(S, dtype=torch.float32, device=f"cuda:{g}") for g in range(G)]
        shard = pkg.SHARD_TILES if mode == "tiles" else pkg.SHARD_SPP
        for g, r in enumerate(rts):
            r.render_accumulate(r.args(nx, ny, ns, True, shard_mode=shard, shard_rank=g, shard_count=G), acc[g].data_ptr())
        # reduce-scatter: every GPU ends up with the sum of its slice, finalises it
        assert L.rt_group_start() == 0
        for g, r in enumerate(rts):
            assert L.rt_reduce_scatter(r._ctx, C.c_void_p(acc[g].data_ptr()), C.c_void_p(sl[g].data_ptr()), S) == 0
        assert L.rt_group_end() == 0
        for g, r in enumerate(rts):
            r.finalize_n(sl[g].data_ptr(), sl[g].data_ptr(), S, ns)
            r.synchronize()
        frame = torch.cat([s.cpu() for s in sl])[:total].view(ny, nx, 3).numpy()
        # reduce onto GPU 0: the same sums
        assert L.rt_group_start() == 0
        for g, r in enumerate(rts):
            assert L.rt_reduce(r._ctx, C.c_void_p(acc[g].data_ptr()), total, 0) == 0
        assert L.rt_group_end() == 0
        fb0 = torch.empty(total, dtype=torch.float32, device="cuda:0")
        rts[0].finalize(acc[0].data_ptr(), fb0.data_ptr(), nx, ny, ns)
        rts[0].synchronize()
        assert np.array_equal(fb0.cpu().numpy().view(np.uint32), frame.reshape(-1).view(np.uint32))
        if mode == "tiles":
            assert np.array_equal(frame.view(np.uint32), ref.view(np.uint32))
        else:
            assert abs(float(frame.mean()) - float(ref.mean())) < 0.01 and not np.array_equal(frame, ref)
    finally:
        for r in rts:
            L.rt_comm_destroy(r._ctx)
            r.close()


def test_host_driven_wavefront_through_get_ray_hit_scatter_reproduces_the_frame(rt, pkg):
    """camera::get_ray, hitTree and material::scatter as separate entry points (rt_camera_get_rays, rt_trace_rays,
    rt_scatter_rays — what include/rt_dropin.h forwards to): a host-driven wavefront over all pixels, drawing from the
    per-pixel streams curand_init(1984 + pixel_index, 0, 0), follows exactly the paths the render kernel follows — same ray
    count, same per-pixel radiance (sky colour recomputed here in float64, hence the 1e-6 tolerance)."""
    nx, ny, n, spl = 64, 48, 488, 30
    rt.create_world(n, 0.1)
    rt.build_octree(spl)
    rt.set_camera(nx, ny)
    import torch
    acc = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    st = rt.render_accumulate(rt.args(nx, ny, 1, True), acc.data_ptr())
    want = acc.cpu().numpy().reshape(-1, 3)
    npix = nx * ny
    states = np.stack([pkg.xorwow_state(1984 + p, 0) for p in range(npix)]).astype(np.uint32)
    jj, ii = np.divmod(np.arange(npix), nx)

    def uniform(s):                       # curand_uniform on the host copy of the states (vectorised XORWOW step)
        t = s[:, 1] ^ (s[:, 1] >> 2)
        s[:, 1], s[:, 2], s[:, 3], s[:, 4] = s[:, 2].copy(), s[:, 3].copy(), s[:, 4].copy(), s[:, 5].copy()
        s[:, 5] = (s[:, 5] ^ (s[:, 5] << 4)) ^ (t ^ (t << 1))
        s[:, 0] += np.uint32(362437)
        x = (s[:, 5] + s[:, 0]).astype(np.uint32)
        return (x.astype(np.float64) * 2.3283064e-10 + 1.16415321826934814453125e-10).astype(np.float32)   # the product is exact: one rounding

    u = ((ii.astype(np.float32) + uniform(states)) / np.float32(nx)).astype(np.float32)
    v = ((jj.astype(np.float32) + uniform(states)) / np.float32(ny)).astype(np.float32)
    org, d = rt.camera_rays(u, v, states)
    att = np.ones((npix, 3), np.float32)
    col = np.zeros((npix, 3), np.float64)
    live = np.arange(npix)
    rays = 0
    for depth in range(50):
        if not len(live):
            break
        rays += len(live)
        idx, t = rt.trace_rays(org[live], d[live], True)
        miss = idx < 0
        if miss.any():
            dm = d[live][miss].astype(np.float64)
            uy = dm[:, 1] / np.sqrt((dm * dm).sum(axis=1))
            tt = 0.5 * (uy + 1.0)
            sky = np.stack([(1 - tt) + tt * 0.5, (1 - tt) + tt * 0.7, (1 - tt) + tt], axis=1)
            col[live[miss]] = att[live[miss]].astype(np.float64) * sky
        hit = ~miss
        if not hit.any():
            live = live[:0]
            break
        h = live[hit]
        sub = np.ascontiguousarray(states[h])
        out = rt.scatter_rays(idx[hit], org[h], d[h], t[hit], sub)
        states[h] = sub
        go = out["scattered"] == 1
        att[h] = (att[h] * out["atten"]).astype(np.float32)
        org[h], d[h] = out["p"], out["dir"]
        live = h[go]
    assert rays == st["rays"]
    ok = np.isclose(col, want.astype(np.float64), rtol=2e-6, atol=1e-7).all(axis=1)
    assert ok.mean() == 1.0, (ok.mean(), np.nonzero(~ok)[0][:10])


def test_dropin_octree_hit_scatter_and_get_ray_members(rt, pkg, O, tmp_path):
    """include/rt_dropin.h: buildOctree returns the reference-layout tree (byte-identical to the oracle's serial build), hitTree
    the oracle's closest hit, material::scatter and camera::get_ray what the library computes for the same inputs."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "octree_dropin")
    lib_dir = os.path.dirname(pkg.LIB_PATH)
    subprocess.run(["g++", "-std=c++17", "-O2", "-I", os.path.join(root, "include"), os.path.join(root, "tests", "dropin", "octree_dropin.cpp"),
                    "-o", exe, f"-L{lib_dir}", "-lrt_b200", f"-Wl,-rpath,{lib_dir}"], check=True)
    n, spl = 488, 30
    sph, _ = O.create_world(n)
    blob, _ = O.build_octree(sph, spl)
    rr = np.random.default_rng(5)
    Q, G = 120, 40
    org = np.stack([rr.uniform(-12, 13, Q), rr.uniform(0.05, 3, Q), rr.uniform(-12, 12, Q)], 1).astype(np.float32)
    dirs = rr.normal(size=(Q, 3)).astype(np.float32)
    dirs[:, 1] = -np.abs(dirs[:, 1])                                  # downwards: most rays hit something
    ss, tt = rr.random(G).astype(np.float32), rr.random(G).astype(np.float32)
    lines = [str(n)] + [" ".join([float(s["cx"]).hex(), float(s["cy"]).hex(), float(s["cz"]).hex(), float(s["radius"]).hex(), str(int(s["mat"])),
                                  float(s["ax"]).hex(), float(s["ay"]).hex(), float(s["az"]).hex(), float(s["param"]).hex()]) for s in sph]
    lines += [str(Q)] + [" ".join(float(x).hex() for x in (*o, *d)) for o, d in zip(org, dirs)]
    lines += [str(G)] + [f"{float(s).hex()} {float(t).hex()} {1984 + k}" for k, (s, t) in enumerate(zip(ss, tt))]
    out = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout.splitlines()
    # the tree
    h = 1469598103934665603
    for byte in blob.tobytes():
        h = ((h ^ byte) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    f = out[0].split()
    assert f[0] == "octree" and int(f[3]) == len(blob.tobytes()) and int(f[4], 16) == h
    # hitTree + scatter against the oracle / the library's batched entry points
    rt.upload_world(sph)
    rt.build_octree(spl)
    gi, gt = rt.trace_rays(org, dirs, True)
    states = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(Q)]).astype(np.uint32)
    hits = np.nonzero(gi >= 0)[0]
    sub = np.ascontiguousarray(states[hits])
    sc = rt.scatter_rays(gi[hits], org[hits], dirs[hits], gt[hits], sub)
    pos = {int(k): q for q, k in enumerate(hits)}
    assert len(hits) > Q // 3
    for k in range(Q):
        oi, ot = O.closest_hit(sph, org[k], dirs[k], blob, spl, True)
        f = out[1 + k].split()
        if oi < 0:
            assert f == ["-1"]
            continue
        assert int(f[0]) == oi and np.float32(float.fromhex(f[1])) == np.float32(ot)
        q = pos[k]
        got_p = [np.float32(float.fromhex(x)) for x in f[2:5]]
        assert got_p == list(sc["p"][q]) and int(f[8]) == int(sc["scattered"][q])
        assert [np.float32(float.fromhex(x)) for x in f[9:12]] == list(sc["atten"][q])
        assert [np.float32(float.fromhex(x)) for x in f[12:15]] == list(sc["dir"][q])
        nrm = np.array([float.fromhex(x) for x in f[5:8]])
        assert abs(np.linalg.norm(nrm) - 1.0) < 2e-3      # (the ground sphere: (p - c) / 1000 in float)
    # get_ray
    rt.set_camera(1200, 800)
    gs = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(G)]).astype(np.uint32)
    co, cd = rt.camera_rays(ss, tt, gs)
    for k in range(G):
        f = out[1 + Q + k].split()
        assert [np.float32(float.fromhex(x)) for x in f[0:3]] == list(co[k]) and [np.float32(float.fromhex(x)) for x in f[3:6]] == list(cd[k])
        assert np.linalg.norm(co[k] - np.array([13, 2, 3], np.float32)) <= 0.05 + 1e-5       # inside the lens disk


@pytest.mark.skipif(_multi_gpu_count() < 2, reason="needs two GPUs")
def test_torch_distributed_nccl_frame_equals_the_one_gpu_frame():
    """multigpu.render_sharded over torch.distributed / NCCL, two ranks (what `bench.py --gpus 2` runs): render on torch's current
    stream, reduce-scatter, per-rank finalise, slices copied into the shared pinned host frame — all without host synchronisation in
    between (round 1 raced here).  With tile shards the assembled frame must be the 1-GPU frame bit for bit; bench.py checks it."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29577",
           os.path.join(root, "bench.py"), "--gpus", "2", "--steps", "2", "--warmup", "3", "--config", "C2", "--shard", "tiles", "--no-cpu-baseline"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    chk = line["e2e"]["frame_check"]
    assert line["n_gpus"] == 2 and chk["sharding"] == "tiles" and chk["identical_to_1gpu_frame"] is True, chk
