"""GPU tier (-m gpu): the USE_FP16 per-ray queries — hitTree / hitable_list::hit, camera::get_ray and material::scatter of the
reference's FP16 build (rt_trace_rays_ex, rt_camera_get_rays_ex, rt_scatter_rays_ex) — the FP16 Octree export, and the
drop-in header compiled with -DUSE_FP16.  Value convention of the FP16 queries: float inputs are rounded to half on entry,
outputs are halves widened to float, so outputs go back in exactly."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RT_ERR_INVALID, RT_ERR_STATE = 10001, 10002
# Per-pixel bound of the wavefront test.  Every path decision and every half value along a path is reproduced exactly; only
# the sky colour of the last ray is recomputed on the host in float64 instead of in half (sky_h: unit_vector with __hdiv, a
# few half roundings), so a pixel's radiance may differ from the frame's by a few units in the last place of its half.
SKY_MAX_HALF_ULPS = 4           # measured on a B200: at most 1.84 over the six scenes below


@pytest.fixture(scope="module")
def rt(pkg):
    r = pkg.RayTracer(0)
    yield r
    r.close()


def _h(x):
    """round to half, widened back to float32 (what the FP16 queries take and give)"""
    return np.asarray(x, dtype=np.float32).astype(np.float16).astype(np.float32)


def _uniform(s):
    """curand_uniform on the host copy of the states (vectorised XORWOW step), as float32"""
    t = s[:, 1] ^ (s[:, 1] >> 2)
    s[:, 1], s[:, 2], s[:, 3], s[:, 4] = s[:, 2].copy(), s[:, 3].copy(), s[:, 4].copy(), s[:, 5].copy()
    s[:, 5] = (s[:, 5] ^ (s[:, 5] << 4)) ^ (t ^ (t << 1))
    s[:, 0] += np.uint32(362437)
    x = (s[:, 5] + s[:, 0]).astype(np.uint32)
    return (x.astype(np.float64) * 2.3283064e-10 + 1.16415321826934814453125e-10).astype(np.float32)   # the product is exact


def _next_draw(state6):
    """curand() of one state {d, v0..v4} without changing it"""
    d, v0, v4 = int(state6[0]), int(state6[1]), int(state6[5])
    m = 0xFFFFFFFF
    t = v0 ^ (v0 >> 2)
    v4 = (v4 ^ ((v4 << 4) & m)) ^ (t ^ ((t << 1) & m))
    return (v4 + d + 362437) & m


def _sky(d):
    """main.cu:68-71 in float64"""
    d = d.astype(np.float64)
    t = 0.5 * (d[:, 1] / np.sqrt((d * d).sum(axis=1)) + 1.0)
    return np.stack([(1 - t) + t * 0.5, (1 - t) + t * 0.7, (1 - t) + t], axis=1)


@pytest.mark.parametrize("n,spl,octree,seed_mode", [
    (488, 30, True, 0),
    (488, 30, False, 0),            # hitable_list::hit over all spheres
    (488, 30, True, 1),             # upstream seeding curand_init(1984, pixel_index, 0)
    (8000, 30, True, 0),
    (20000, 30, True, 0),           # cells overflow: the reference drops entries ("Leaf nodes full")
    (100000, 300, True, 0),
])
def test_host_driven_fp16_wavefront_reproduces_the_fp16_frame(rt, pkg, n, spl, octree, seed_mode):
    """camera::get_ray, hitTree / hitable_list::hit and material::scatter of the FP16 build as separate entry points: a host-driven
    wavefront over all pixels, drawing from the per-pixel streams, follows exactly the paths k_render_h follows (same ray count,
    same absorbed pixels) and reaches the frame's radiance up to the sky colour, which it recomputes in float64."""
    import torch
    F16 = pkg.PREC_FP16
    nx, ny = 64, 32                 # powers of two: the half division of main.cu:104-106 is exact, so numpy reproduces it
    rt.create_world(n, 0.1, precision=F16)
    if octree:
        st = rt.build_octree(spl, precision=F16)
        if n == 20000:
            assert st["dropped_full"] > 0
    rt.set_camera(nx, ny)
    acc = torch.empty((ny, nx, 3), dtype=torch.float32, device="cuda")
    stats = rt.render_accumulate(rt.args(nx, ny, 1, octree, seed_mode=seed_mode, precision=F16), acc.data_ptr())
    want = acc.cpu().numpy().reshape(-1, 3).astype(np.float64)
    npix = nx * ny
    if seed_mode == pkg.SEED_HEAD:
        states = np.stack([pkg.xorwow_state(1984 + p, 0) for p in range(npix)]).astype(np.uint32)
    else:
        states = np.stack([pkg.xorwow_state(1984, p) for p in range(npix)]).astype(np.uint32)
    jj, ii = np.divmod(np.arange(npix), nx)
    # k_render_h: real_t(i + U) / real_t(nx) — the sum in float, rounded to half, then __hdiv (exact for a power-of-two divisor)
    u = _h(_h(ii.astype(np.float32) + _uniform(states)) / np.float32(nx))
    v = _h(_h(jj.astype(np.float32) + _uniform(states)) / np.float32(ny))
    org, d = rt.camera_rays(u, v, states, precision=F16)
    att = np.ones((npix, 3), np.float16)
    col = np.zeros((npix, 3), np.float64)
    live = np.arange(npix)
    rays = 0
    for depth in range(50):
        if not len(live):
            break
        rays += len(live)
        idx, t = rt.trace_rays(org[live], d[live], octree, precision=F16)
        miss = idx < 0
        if miss.any():
            lm = live[miss]
            col[lm] = att[lm].astype(np.float64) * _sky(d[lm])
        hit = ~miss
        h = live[hit]
        if not len(h):
            break
        sub = np.ascontiguousarray(states[h])
        out = rt.scatter_rays(idx[hit], org[h], d[h], t[hit], sub, precision=F16)
        states[h] = sub
        assert (out["scattered"] >= 0).all()
        go = out["scattered"] == 1
        hg = h[go]
        att[hg] = att[hg] * out["atten"][go].astype(np.float16)          # a product of two halves, rounded once (__hmul)
        org[hg], d[hg] = out["p"][go], out["dir"][go]
        live = hg
    assert rays == stats["rays"]
    zero_frame, zero_host = (want == 0).all(axis=1), (col == 0).all(axis=1)
    assert np.array_equal(zero_frame, zero_host), np.nonzero(zero_frame != zero_host)[0][:10]
    ulp = np.spacing(np.abs(want).astype(np.float16)).astype(np.float64)
    err = np.abs(col - want) / ulp
    print(f"n={n} octree={octree} seed={seed_mode}: rays={rays} absorbed={int(zero_frame.sum())} max |host - frame| = {err.max():.2f} half ulps")
    assert err.max() <= SKY_MAX_HALF_ULPS, (err.max(), np.unravel_index(np.argmax(err), err.shape))


def _rays(rr, sph, count):
    """random origins, aimed near random spheres (the FP16 world has no ground: r * r overflows half, so a ray aimed anywhere
    else misses)"""
    org = _h(np.stack([rr.uniform(-12, 13, count), rr.uniform(0.05, 3, count), rr.uniform(-12, 12, count)], 1))
    k = rr.integers(1, len(sph), count)
    target = np.stack([sph["cx"][k], sph["cy"][k], sph["cz"][k]], 1) + rr.normal(scale=0.05, size=(count, 3))
    return org, _h(target - org)


def _chunked(fn, count, chunk):
    parts = [fn(slice(a, min(a + chunk, count))) for a in range(0, count, chunk)]
    return [np.concatenate(p) for p in zip(*parts)]


def _same(a, b):
    return np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32))


@pytest.mark.parametrize("n,spl,octree", [(8000, 30, True), (488, 30, False)])
def test_fp16_queries_do_not_depend_on_the_batch(rt, pkg, n, spl, octree):
    """The same FP16 inputs in one batch, in reverse order and in chunks of 1, 31, 33 and 1 000 give bit-identical outputs —
    trace (the warp shares every ray's scan), camera and scatter — and every output is a half widened to float."""
    F16 = pkg.PREC_FP16
    rt.create_world(n, 0.1, precision=F16)
    if octree:
        rt.build_octree(spl, precision=F16)
    rt.set_camera(96, 64)
    rr = np.random.default_rng(n)
    R = 1200
    org, dirs = _rays(rr, rt.spheres(), R)
    idx, t = rt.trace_rays(org, dirs, octree, precision=F16)
    assert (idx >= 0).sum() > R // 3 and _same(t, _h(t))
    ri, rtt = rt.trace_rays(org[::-1], dirs[::-1], octree, precision=F16)
    assert _same(ri[::-1], idx) and _same(rtt[::-1], t)
    for chunk in (1, 31, 33, 1000):
        ci, ct = _chunked(lambda s: rt.trace_rays(org[s], dirs[s], octree, precision=F16), R, chunk)
        assert _same(ci, idx) and _same(ct, t), chunk

    G = 300
    ss, tt = rr.random(G), rr.random(G)
    st0 = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(G)]).astype(np.uint32)

    def cam(s, rev=False):
        st = np.array(st0[s][::-1] if rev else st0[s], copy=True)       # advanced in place
        o, d = rt.camera_rays(ss[s][::-1] if rev else ss[s], tt[s][::-1] if rev else tt[s], st, precision=F16)
        return (o[::-1], d[::-1], st[::-1]) if rev else (o, d, st)
    co, cd, cs = cam(slice(0, G))
    assert _same(co, _h(co)) and _same(cd, _h(cd)) and not np.array_equal(cs, st0)
    for got in [cam(slice(0, G), rev=True)] + [_chunked(cam, G, c) for c in (1, 31, 33, 1000)]:
        assert _same(got[0], co) and _same(got[1], cd) and np.array_equal(got[2], cs)

    hits = np.nonzero(idx >= 0)[0]
    si = idx[hits].copy()
    si[::97] = -1                                   # not a sphere: scattered = -1, state untouched
    H = len(hits)
    sst0 = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(H)]).astype(np.uint32)

    def scat(s, rev=False):
        pick = (lambda a: np.array(a[s][::-1], copy=True)) if rev else (lambda a: np.array(a[s], copy=True))
        st = pick(sst0)
        out = rt.scatter_rays(pick(si), pick(org[hits]), pick(dirs[hits]), pick(t[hits]), st, precision=F16)
        res = [out[k] for k in ("p", "normal", "dir", "atten", "scattered")] + [st]
        return [r[::-1] for r in res] if rev else res
    base = scat(slice(0, H))
    assert (base[4][::97] == -1).all() and np.array_equal(base[5][::97], sst0[::97])
    assert set(np.unique(base[4][base[4] >= 0])) <= {0, 1} and (base[4] == 1).sum() > H // 2
    for k in range(4):
        assert _same(base[k], _h(base[k]))
    for got in [scat(slice(0, H), rev=True)] + [_chunked(scat, H, c) for c in (1, 31, 33, 1000)]:
        for a, b in zip(got, base):
            assert _same(a, b)


def test_fp32_ex_entry_points_are_the_fp32_ones(rt, pkg):
    """With RT_PREC_FP32 the _ex entry points return what the entry points without a precision argument return."""
    L = rt.L
    rt.create_world(8000, 0.1)
    rt.build_octree(30)
    rt.set_camera(120, 80)
    rr = np.random.default_rng(7)
    R = 400
    org = np.stack([rr.uniform(-12, 13, R), rr.uniform(0.05, 3, R), rr.uniform(-12, 12, R)], 1).astype(np.float32)
    dirs = rr.normal(size=(R, 3)).astype(np.float32)
    for octree in (True, False):
        a_i, a_t = np.zeros(R, np.int32), np.zeros(R, np.float32)
        assert L.rt_trace_rays(rt._ctx, int(octree), R, org.ctypes.data, dirs.ctypes.data, a_i.ctypes.data, a_t.ctypes.data) == 0
        b_i, b_t = rt.trace_rays(org, dirs, octree, precision=pkg.PREC_FP32)
        assert _same(a_i, b_i) and _same(a_t, b_t)
    s, t = rr.random(R).astype(np.float32), rr.random(R).astype(np.float32)
    st_a = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(R)]).astype(np.uint32)
    st_b = st_a.copy()
    o_a, d_a = np.zeros((R, 3), np.float32), np.zeros((R, 3), np.float32)
    assert L.rt_camera_get_rays(rt._ctx, R, s.ctypes.data, t.ctypes.data, st_a.ctypes.data, o_a.ctypes.data, d_a.ctypes.data) == 0
    o_b, d_b = rt.camera_rays(s, t, st_b, precision=pkg.PREC_FP32)
    assert _same(o_a, o_b) and _same(d_a, d_b) and np.array_equal(st_a, st_b)
    gi, gt = rt.trace_rays(org, dirs, True)
    hits = np.nonzero(gi >= 0)[0]
    st_a = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(len(hits))]).astype(np.uint32)
    st_b = st_a.copy()
    a = {k: np.zeros((len(hits), 3), np.float32) for k in ("p", "normal", "dir", "atten")}
    a["scattered"] = np.zeros(len(hits), np.int32)
    hi, ho, hd, ht = (np.ascontiguousarray(x[hits]) for x in (gi, org, dirs, gt))
    assert L.rt_scatter_rays(rt._ctx, len(hits), hi.ctypes.data, ho.ctypes.data, hd.ctypes.data, ht.ctypes.data, st_a.ctypes.data,
                             a["p"].ctypes.data, a["normal"].ctypes.data, a["dir"].ctypes.data, a["atten"].ctypes.data,
                             a["scattered"].ctypes.data) == 0
    b = rt.scatter_rays(hi, ho, hd, ht, st_b, precision=pkg.PREC_FP32)
    assert all(_same(a[k], b[k]) for k in a) and np.array_equal(st_a, st_b)


# ---- the FP16 Octree export -----------------------------------------------------------------------------------------------------

def _parse_octree(blob, spl, fp16):
    """Octree (acceleration_structure.h:23-61): nodes[585] {level, AABB, children[8]}, leaves[4097] {indices[spl], count},
    nodeCount, leafCount.  AABB: six floats (60-byte nodes) or, under USE_FP16, six halves (48-byte nodes)."""
    nb = 48 if fp16 else 60
    raw = blob.tobytes()
    assert len(raw) == 585 * nb + 4097 * (spl + 1) * 4 + 8
    nodes = np.frombuffer(raw[:585 * nb], dtype=np.uint8).reshape(585, nb)
    level = np.ascontiguousarray(nodes[:, :4]).view("<i4")[:, 0]
    if fp16:
        box = np.ascontiguousarray(nodes[:, 4:16]).view("<f2").astype(np.float32)
        children = np.ascontiguousarray(nodes[:, 16:48]).view("<i4")
    else:
        box = np.ascontiguousarray(nodes[:, 4:28]).view("<f4")
        children = np.ascontiguousarray(nodes[:, 28:60]).view("<i4")
    leaves = np.frombuffer(raw[585 * nb:585 * nb + 4097 * (spl + 1) * 4], dtype="<i4").reshape(4097, spl + 1)
    node_count, leaf_count = (int(x) for x in np.frombuffer(raw[-8:], dtype="<i4"))
    return level, box, children, leaves, node_count, leaf_count


def _existing_nodes(cell_start):
    cs = cell_start.astype(np.int64)
    per = lambda k: int((cs[k::k][:512 // k] > cs[0:512:k]).sum())      # nodes whose subtree received an entry, k cells each
    return 1 + per(64) + per(8) + per(1)


@pytest.mark.parametrize("n,spl", [(488, 30), (8000, 30)])
def test_fp16_octree_export_matches_the_reference_fp16_build(rt, pkg, golden_dir, n, spl):
    """The exported USE_FP16 Octree: its level-3 node lows and their bucket chains are the ones the reference's FP16 build
    produced, nodeCount is the number of nodes that exist, and every child's AABB is its parent's octant."""
    gold = np.load(os.path.join(golden_dir, "ref_cuda", f"n{n}_spl{spl}_fp16_cells.npz"))
    rt.create_world(n, 0.1, precision=pkg.PREC_FP16)
    rt.build_octree(spl, precision=pkg.PREC_FP16)
    blob = rt.export_octree()
    level, box, children, leaves, node_count, leaf_count = _parse_octree(blob, spl, True)
    assert node_count == _existing_nodes(rt.debug_tree()["cell_start"].view(np.uint32))
    cells = {}
    for k in range(node_count):
        if level[k] == 3:
            lst = []
            for c in children[k]:
                if c == 0:
                    break
                assert 1 <= c < leaf_count
                lst.extend(int(x) for x in leaves[c, :leaves[c, spl]])
            cells[tuple(float(x) for x in box[k, :3])] = lst
        else:
            lo, hi = box[k, :3], box[k, 3:]
            mid = (lo + hi) / 2
            for c, ch in enumerate(children[k]):
                if ch == 0:
                    continue
                bits = np.array([c >> 2, (c >> 1) & 1, c & 1]).astype(bool)
                assert level[ch] == level[k] + 1
                assert np.array_equal(box[ch, :3], np.where(bits, mid, lo)) and np.array_equal(box[ch, 3:], np.where(bits, hi, mid)), (k, c)
    want = {tuple(float(x) for x in low): [int(x) for x in gold["idx"][gold["start"][k]:gold["start"][k + 1]]]
            for k, low in enumerate(gold["low"])}
    assert cells == want
    assert (level[node_count:] == 0).all() and (box[node_count:] == 0).all()


def test_fp16_octree_export_is_the_fp32_layout_with_half_boxes(rt, pkg):
    """A scene whose FP16 and FP32 cell memberships are identical (centres well inside their cells, every value exact in half):
    the FP16 blob's integer fields equal the FP32 blob's, and its AABBs are the FP32 AABBs rounded to half."""
    rr = np.random.default_rng(11)
    N = 3000
    sph = np.zeros(N, dtype=pkg.SPHERE_DTYPE)
    sph[0] = (0, -1000, -1, 1000, pkg.MAT_LAMBERTIAN, 0.5, 0.5, 0.5, 0)
    ix, iy, iz = rr.integers(0, 8, N), rr.integers(0, 8, N), rr.integers(0, 8, N)
    ix[:600], iy[:600], iz[:600] = 3, 3, 3                 # more than 8 * SPL in one cell: the reference drops the rest
    jit = lambda: np.round(rr.uniform(-1, 1, N) * 64) / 64
    sph["cx"][1:] = (-11 + 2.75 * (ix + 0.5) + jit())[1:]
    sph["cy"][1:] = (0.25 * (iy + 0.5))[1:]
    sph["cz"][1:] = (-11 + 2.75 * (iz + 0.5) + jit())[1:]
    sph["radius"][1:] = 0.0625
    sph["mat"][1:] = pkg.MAT_LAMBERTIAN
    sph["ax"][1:] = sph["ay"][1:] = sph["az"][1:] = 0.5
    assert all(np.array_equal(sph[f], _h(sph[f])) for f in ("cx", "cy", "cz", "radius"))
    spl = 30
    rt.upload_world(sph)
    rt.build_octree(spl, precision=pkg.PREC_FP32)
    t32 = rt.debug_tree()
    b32 = rt.export_octree()
    rt.build_octree(spl, precision=pkg.PREC_FP16)
    t16 = rt.debug_tree()
    b16 = rt.export_octree()
    assert np.array_equal(t32["cell_start"], t16["cell_start"]) and np.array_equal(t32["cell_list"], t16["cell_list"])
    assert int(np.diff(t32["cell_start"].view(np.uint32).astype(np.int64)).max()) > 8 * spl      # some buckets overflow too
    p32, p16 = _parse_octree(b32, spl, False), _parse_octree(b16, spl, True)
    for k in (0, 2, 3, 4, 5):                             # level, children, leaves, nodeCount, leafCount
        assert np.array_equal(p32[k], p16[k]), k
    assert np.array_equal(p16[1], _h(p32[1]))
    assert b16.size == rt.L.rt_octree_reference_bytes_ex(spl, pkg.PREC_FP16)


# ---- the drop-in header under -DUSE_FP16 ------------------------------------------------------------------------------------------

def test_dropin_use_fp16_members_match_the_library(rt, pkg, tmp_path):
    """include/rt_dropin.h built with -DUSE_FP16: buildOctree returns the FP16 build's tree in its layout, hitTree and
    material::scatter answer what rt_trace_rays_ex / rt_scatter_rays_ex(RT_PREC_FP16) answer (rec.t, rec.p, rec.normal are the
    library's half values), camera::get_ray what rt_camera_get_rays_ex(RT_PREC_FP16) answers — bit for bit, on half inputs."""
    F16 = pkg.PREC_FP16
    exe = str(tmp_path / "fp16_dropin")
    lib_dir = os.path.dirname(pkg.LIB_PATH)
    subprocess.run(["g++", "-std=c++17", "-O2", "-DUSE_FP16", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "dropin", "fp16_dropin.cpp"),
                    "-o", exe, f"-L{lib_dir}", "-lrt_b200", f"-Wl,-rpath,{lib_dir}"], check=True)
    n, spl = 488, 30
    rt.create_world(n, 0.1, precision=F16)
    sph = rt.spheres()                                    # the FP16 world: every value already a half
    rr = np.random.default_rng(5)
    Q, G = 160, 40
    org, dirs = _rays(rr, sph, Q)
    ss, tt = _h(rr.random(G)), _h(rr.random(G))
    hx = lambda x: float(x).hex()
    lines = [str(n)] + [" ".join([hx(s["cx"]), hx(s["cy"]), hx(s["cz"]), hx(s["radius"]), str(int(s["mat"])), hx(s["ax"]), hx(s["ay"]),
                                  hx(s["az"]), hx(s["param"])]) for s in sph]
    lines += [str(Q)] + [" ".join(hx(x) for x in (*o, *d)) for o, d in zip(org, dirs)]
    lines += [str(G)] + [f"{hx(s)} {hx(t)} {1984 + k}" for k, (s, t) in enumerate(zip(ss, tt))]
    out = subprocess.run([exe], input="\n".join(lines) + "\n", capture_output=True, text=True, check=True).stdout.splitlines()
    f32 = lambda s: np.float32(float.fromhex(s))
    # the tree
    rt.upload_world(sph)
    rt.build_octree(spl, precision=F16)
    blob = rt.export_octree()
    h = 1469598103934665603
    for byte in blob.tobytes():
        h = ((h ^ byte) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    _, _, _, _, node_count, leaf_count = _parse_octree(blob, spl, True)
    assert out[0].split() == ["octree", str(node_count), str(leaf_count), "536116", f"{h:016x}"]
    # hitTree + scatter
    gi, gt = rt.trace_rays(org, dirs, True, precision=F16)
    hits = np.nonzero(gi >= 0)[0]
    assert len(hits) > Q // 3
    states = np.stack([pkg.xorwow_state(1984 + int(k), 0) for k in hits]).astype(np.uint32)
    sc = rt.scatter_rays(gi[hits], org[hits], dirs[hits], gt[hits], states, precision=F16)
    pos = {int(k): q for q, k in enumerate(hits)}
    for k in range(Q):
        f = out[1 + k].split()
        if gi[k] < 0:
            assert f == ["-1"]
            continue
        q = pos[k]
        assert int(f[0]) == gi[k] and f32(f[1]) == gt[k]
        assert [f32(x) for x in f[2:5]] == list(sc["p"][q]) and [f32(x) for x in f[5:8]] == list(sc["normal"][q])
        assert int(f[8]) == int(sc["scattered"][q] == 1)
        if f[8] == "1":
            assert [f32(x) for x in f[9:12]] == list(sc["p"][q])
            assert [f32(x) for x in f[12:15]] == list(sc["atten"][q]) and [f32(x) for x in f[15:18]] == list(sc["dir"][q])
            assert int(f[18]) == _next_draw(states[q])
    # get_ray
    desc = pkg.CameraDesc((13, 2, 3), (0, 0, 0), (0, 1, 0), 30.0, 1.5, 0.1, 10.0)
    rt.set_camera(1200, 800, desc)
    gs = np.stack([pkg.xorwow_state(1984 + k, 0) for k in range(G)]).astype(np.uint32)
    co, cd = rt.camera_rays(ss, tt, gs, precision=F16)
    for k in range(G):
        f = out[1 + Q + k].split()
        assert [f32(x) for x in f[0:3]] == list(co[k]) and [f32(x) for x in f[3:6]] == list(cd[k])
        assert int(f[6]) == _next_draw(gs[k])


# ---- errors --------------------------------------------------------------------------------------------------------------------

def test_fp16_query_errors(rt, pkg):
    L = rt.L
    one = np.zeros(8, np.float32)
    oi, st6 = np.zeros(8, np.int32), np.ones((1, 6), np.uint32)
    p = lambda a: a.ctypes.data
    trace = lambda r, octree, prec: L.rt_trace_rays_ex(r._ctx, octree, prec, 1, p(one), p(one), p(oi), p(one))
    camera = lambda r, prec: L.rt_camera_get_rays_ex(r._ctx, prec, 1, p(one), p(one), p(st6), p(one), p(one))
    scatter = lambda r, prec: L.rt_scatter_rays_ex(r._ctx, prec, 1, p(oi), p(one), p(one), p(one), p(st6), p(one), p(one), p(one), p(one), p(oi))
    # no scene, no camera, no octree
    fresh = pkg.RayTracer(0)
    try:
        assert trace(fresh, 0, pkg.PREC_FP16) == RT_ERR_STATE
        assert scatter(fresh, pkg.PREC_FP16) == RT_ERR_STATE
        assert camera(fresh, pkg.PREC_FP16) == RT_ERR_STATE
        fresh.create_world(488, 0.1, precision=pkg.PREC_FP16)
        assert trace(fresh, 1, pkg.PREC_FP16) == RT_ERR_STATE            # no octree built
    finally:
        fresh.close()
    # unknown precision
    rt.create_world(488, 0.1)
    rt.set_camera(64, 32)
    rt.build_octree(30)
    for prec in (2, -1):
        assert trace(rt, 0, prec) == RT_ERR_INVALID and camera(rt, prec) == RT_ERR_INVALID and scatter(rt, prec) == RT_ERR_INVALID
    # an octree query in one precision on a tree built for the other
    assert trace(rt, 1, pkg.PREC_FP16) == RT_ERR_STATE
    assert b"other precision" in L.rt_last_error(rt._ctx)
    assert trace(rt, 0, pkg.PREC_FP16) == 0                              # the flat list needs no tree
    rt.build_octree(30, precision=pkg.PREC_FP16)
    assert trace(rt, 1, pkg.PREC_FP32) == RT_ERR_STATE
    assert trace(rt, 1, pkg.PREC_FP16) == 0
    with pytest.raises(pkg.RtError, match="other precision"):
        rt.trace_rays(one[:3].reshape(1, 3), one[:3].reshape(1, 3), True)
