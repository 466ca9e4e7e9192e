"""dd2360-raytracing_b200 — host-side mirror of the reference's render path over librt_b200.so (sm_100a CUDA).

The compute lives in hand-written CUDA behind the C ABI of include/rt_abi.h; this module only binds it with
ctypes and mirrors the call sequence of the reference's main() (main.cu:347-477):

    rt = RayTracer(device=0)
    rt.create_world(n=488, radius=0.1)          # rand_init + create_world          main.cu:388,399
    rt.build_octree(spheres_per_leaf=30)        # D2H + buildOctree + H2D           main.cu:405-415
    fb = rt.render(nx, ny, ns, use_octree=True) # render_init + render              main.cu:424-429
    ppm = format_ppm(fb)                        # output_to_stream                  main.cu:321-333

There is NO CPU fallback: importing works anywhere (so CPU-only CI can check the ABI surface), but every compute
call needs the built library and a CUDA device and raises otherwise.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librt_b200.so")
LIB_COUNTERS_PATH = os.path.join(HERE, "librt_b200_counters.so")   # same kernels + work counters (roofline inputs)
INCLUDE_DIR = os.path.normpath(os.path.join(HERE, "..", "include"))

MAT_NONE, MAT_LAMBERTIAN, MAT_METAL, MAT_DIELECTRIC = -1, 0, 1, 2
SEED_HEAD, SEED_UPSTREAM = 0, 1
SHARD_NONE, SHARD_TILES, SHARD_SPP = 0, 1, 2
PREC_FP32, PREC_FP16 = 0, 1

SPHERE_DTYPE = np.dtype(
    [("cx", "<f4"), ("cy", "<f4"), ("cz", "<f4"), ("radius", "<f4"), ("mat", "<i4"),
     ("ax", "<f4"), ("ay", "<f4"), ("az", "<f4"), ("param", "<f4")]
)

# every symbol include/rt_abi.h declares (tests check the library exports exactly these)
ABI_SYMBOLS = [
    "rt_abi_version", "rt_create", "rt_destroy", "rt_last_error", "rt_set_stream", "rt_device_info",
    "rt_scene_generate", "rt_scene_generate_ex", "rt_scene_upload", "rt_scene_download", "rt_scene_size", "rt_camera_set", "rt_camera_get", "rt_camera_get_half",
    "rt_octree_build", "rt_octree_build_ex", "rt_octree_reference_bytes", "rt_octree_reference_bytes_ex", "rt_octree_export_reference", "rt_octree_debug_read", "rt_xorwow_state", "rt_debug_counters", "rt_trace_rays", "rt_camera_get_rays", "rt_scatter_rays",
    "rt_trace_rays_ex", "rt_camera_get_rays_ex", "rt_scatter_rays_ex",
    "rt_render_accumulate", "rt_last_render_stats", "rt_render_progressive", "rt_finalize", "rt_finalize_n", "rt_finalize_ex", "rt_render", "rt_render_to_host", "rt_render_pixels", "rt_format_ppm",
    "rt_ppm_format", "rt_ppm_read", "rt_render_to_ppm",
    "rt_ffma_peak", "rt_hfma2_peak", "rt_malloc", "rt_free", "rt_memcpy_to_host", "rt_synchronize", "rt_kernel_name",
    "rt_comm_get_unique_id", "rt_comm_init_rank", "rt_comm_init_all", "rt_comm_attach", "rt_comm_destroy", "rt_comm_rank", "rt_comm_size",
    "rt_group_start", "rt_group_end", "rt_reduce", "rt_reduce_scatter", "rt_broadcast",
]


class OctreeStats(C.Structure):
    _fields_ = [("node_count", C.c_int32), ("leaf_count", C.c_int32), ("entries", C.c_int64),
                ("dropped_full", C.c_int64), ("dropped_outside", C.c_int64), ("fine_voxels", C.c_int64),
                ("fine_refs", C.c_int64), ("build_ms", C.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class RenderArgs(C.Structure):
    _fields_ = [("nx", C.c_int32), ("ny", C.c_int32), ("ns", C.c_int32), ("max_depth", C.c_int32),
                ("use_octree", C.c_int32), ("seed_mode", C.c_int32), ("shard_mode", C.c_int32),
                ("shard_rank", C.c_int32), ("shard_count", C.c_int32), ("precision", C.c_int32), ("tune", C.c_int32 * 6)]


class RenderStats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("paths", C.c_uint64), ("sphere_tests", C.c_uint64), ("node_tests", C.c_uint64),
                ("kernel_ms", C.c_float), ("launches", C.c_int32), ("kernel_id", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}
        d["kernel"] = load_library().rt_kernel_name(self.kernel_id).decode()
        return d


class CameraDesc(C.Structure):
    _fields_ = [("lookfrom", C.c_float * 3), ("lookat", C.c_float * 3), ("vup", C.c_float * 3),
                ("vfov", C.c_float), ("aspect", C.c_float), ("aperture", C.c_float), ("focus_dist", C.c_float)]


class RtError(RuntimeError):
    pass


_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """dlopen librt_b200.so and declare the ABI.  Fails loudly when the extension has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise RtError(f"{p} is missing: build it with `python dd2360-raytracing_b200/build.py` "
                      f"(nvcc, sm_100a). There is no CPU fallback.")
    L = C.CDLL(p)
    vp, i32, f32, sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
    sig = {
        "rt_abi_version": (i32, []),
        "rt_create": (i32, [i32, C.POINTER(vp)]),
        "rt_destroy": (None, [vp]),
        "rt_last_error": (C.c_char_p, [vp]),
        "rt_set_stream": (i32, [vp, vp]),
        "rt_kernel_name": (C.c_char_p, [i32]),
        "rt_device_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(sz)]),
        "rt_scene_generate": (i32, [vp, i32, f32]),
        "rt_scene_generate_ex": (i32, [vp, i32, f32, i32]),
        "rt_scene_upload": (i32, [vp, vp, i32]),
        "rt_scene_download": (i32, [vp, vp, i32]),
        "rt_scene_size": (i32, [vp]),
        "rt_camera_set": (i32, [vp, C.POINTER(CameraDesc), i32, i32]),
        "rt_camera_get": (i32, [vp, vp]),
        "rt_camera_get_half": (i32, [vp, i32, i32, vp]),
        "rt_octree_build": (i32, [vp, i32, C.POINTER(OctreeStats)]),
        "rt_octree_build_ex": (i32, [vp, i32, i32, C.POINTER(OctreeStats)]),
        "rt_octree_reference_bytes": (sz, [i32]),
        "rt_octree_reference_bytes_ex": (sz, [i32, i32]),
        "rt_octree_export_reference": (i32, [vp, vp, sz]),
        "rt_octree_debug_read": (sz, [vp, i32, vp, sz]),
        "rt_xorwow_state": (i32, [C.c_uint64, C.c_uint64, vp]),
        "rt_debug_counters": (i32, [vp, vp]),
        "rt_trace_rays": (i32, [vp, i32, i32, vp, vp, vp, vp]),
        "rt_camera_get_rays": (i32, [vp, i32, vp, vp, vp, vp, vp]),
        "rt_scatter_rays": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "rt_trace_rays_ex": (i32, [vp, i32, i32, i32, vp, vp, vp, vp]),
        "rt_camera_get_rays_ex": (i32, [vp, i32, i32, vp, vp, vp, vp, vp]),
        "rt_scatter_rays_ex": (i32, [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "rt_render_accumulate": (i32, [vp, C.POINTER(RenderArgs), vp, C.POINTER(RenderStats)]),
        "rt_last_render_stats": (i32, [vp, C.POINTER(RenderStats)]),
        "rt_render_progressive": (i32, [vp, C.POINTER(RenderArgs), vp, vp, i32, C.POINTER(RenderStats)]),
        "rt_finalize": (i32, [vp, vp, vp, i32, i32, i32]),
        "rt_finalize_n": (i32, [vp, vp, vp, sz, i32]),
        "rt_finalize_ex": (i32, [vp, vp, vp, sz, i32, i32]),
        "rt_render": (i32, [vp, C.POINTER(RenderArgs), vp, C.POINTER(RenderStats)]),
        "rt_render_to_host": (i32, [vp, C.POINTER(RenderArgs), vp, C.POINTER(RenderStats)]),
        "rt_render_pixels": (i32, [vp, C.POINTER(RenderArgs), vp, i32, vp, i32, C.POINTER(RenderStats)]),
        "rt_format_ppm": (sz, [vp, i32, i32, vp, sz]),
        "rt_ppm_format": (i32, [vp, vp, i32, i32, C.POINTER(sz)]),
        "rt_ppm_read": (i32, [vp, vp, sz]),
        "rt_render_to_ppm": (i32, [vp, C.POINTER(RenderArgs), C.POINTER(RenderStats), C.POINTER(sz)]),
        "rt_ffma_peak": (i32, [vp, C.POINTER(f32), C.POINTER(f32)]),
        "rt_hfma2_peak": (i32, [vp, C.POINTER(f32), C.POINTER(f32)]),
        "rt_malloc": (i32, [vp, sz, C.POINTER(vp)]),
        "rt_free": (i32, [vp, vp]),
        "rt_memcpy_to_host": (i32, [vp, vp, vp, sz]),
        "rt_synchronize": (i32, [vp]),
        "rt_comm_get_unique_id": (i32, [vp]),
        "rt_comm_init_rank": (i32, [vp, vp, i32, i32]),
        "rt_comm_init_all": (i32, [C.POINTER(vp), i32]),
        "rt_comm_attach": (i32, [vp, vp, i32, i32]),
        "rt_comm_destroy": (i32, [vp]),
        "rt_comm_rank": (i32, [vp]),
        "rt_comm_size": (i32, [vp]),
        "rt_group_start": (i32, []),
        "rt_group_end": (i32, []),
        "rt_reduce": (i32, [vp, vp, sz, i32]),
        "rt_reduce_scatter": (i32, [vp, vp, vp, sz]),
        "rt_broadcast": (i32, [vp, vp, sz, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = L
    return L


def format_ppm(fb: np.ndarray) -> bytes:
    """output_to_stream (main.cu:321-333): P3 text, byte-identical to the reference writer."""
    L = load_library()
    fb = np.ascontiguousarray(fb, dtype=np.float32)
    ny, nx, _ = fb.shape
    need = L.rt_format_ppm(fb.ctypes.data, nx, ny, None, 0)
    buf = C.create_string_buffer(need)
    L.rt_format_ppm(fb.ctypes.data, nx, ny, buf, need)
    return buf.raw[:need]


def xorwow_state(seed: int, subsequence: int) -> np.ndarray:
    """{d, v0..v4} after curand_init(seed, subsequence, 0), from the library's own skip-ahead matrices (host side)."""
    out = np.zeros(6, dtype=np.uint32)
    rc = load_library().rt_xorwow_state(seed, subsequence, out.ctypes.data)
    if rc != 0:
        raise RtError(f"rt_xorwow_state failed ({rc})")
    return out


def window_pixels(nx: int, ny: int, i0: int, i1: int, j0: int, j1: int) -> np.ndarray:
    """Pixel indices j*nx + i of the rectangle i0 <= i < i1, j0 <= j < j1 (the frame region fb[j0:j1, i0:i1]) for
    RayTracer.render_pixels: every pixel once, in 8x4 tiles laid from the rectangle's corner (tiles row by row, pixels row by
    row inside a tile), so that a warp's 32 entries are neighbours in the image as they are in the frame's queue."""
    if not (0 <= i0 < i1 <= nx and 0 <= j0 < j1 <= ny):
        raise ValueError(f"window ({i0}, {i1}, {j0}, {j1}) is empty or outside the {nx}x{ny} frame")
    tx, ty = (i1 - i0 + 7) // 8, (j1 - j0 + 3) // 4
    t_y, t_x, y, x = np.meshgrid(np.arange(ty), np.arange(tx), np.arange(4), np.arange(8), indexing="ij")
    i, j = i0 + t_x * 8 + x, j0 + t_y * 4 + y
    keep = (i < i1) & (j < j1)
    return (j[keep].astype(np.int64) * nx + i[keep]).astype(np.uint32)


def quantise(fb: np.ndarray) -> np.ndarray:
    """int(255.99 * channel) in PPM row order (top row first), as uint8 [ny, nx, 3]."""
    q = (255.99 * fb.astype(np.float64)).astype(np.int64)
    return np.clip(q[::-1], 0, 255).astype(np.uint8)


class RayTracer:
    """One context per GPU: mirrors the reference's main() call sequence over the C ABI."""

    def __init__(self, device: int = 0, instrumented: bool = False):
        self.L = load_library(LIB_COUNTERS_PATH) if instrumented else load_library()
        self._ctx = C.c_void_p()
        rc = self.L.rt_create(device, C.byref(self._ctx))
        if rc != 0:
            raise RtError(f"rt_create(device={device}) failed with code {rc}: no usable CUDA device "
                          f"(this library has no CPU fallback)")
        self.device = device
        self.n = 0
        self.spl = None
        self.octree_precision = PREC_FP32

    # -- plumbing --
    def _ck(self, rc: int, what: str):
        if rc != 0:
            msg = self.L.rt_last_error(self._ctx)
            raise RtError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def close(self):
        if self._ctx:
            self.L.rt_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_handle: int | None):
        """Launch on the given cudaStream_t.  None = the context's own (blocking) stream; 0 — what
        torch.cuda.current_stream().cuda_stream returns for the default stream — selects the LEGACY DEFAULT stream
        (cudaStreamLegacy), so that the library's kernels are ordered with torch's and NCCL's work on it."""
        CUDA_STREAM_LEGACY = 1
        h = 0 if cuda_stream_handle is None else (cuda_stream_handle or CUDA_STREAM_LEGACY)
        self._ck(self.L.rt_set_stream(self._ctx, C.c_void_p(h)), "rt_set_stream")


    def device_info(self):
        sm, clk, mem = C.c_int(), C.c_int(), C.c_size_t()
        self._ck(self.L.rt_device_info(self._ctx, C.byref(sm), C.byref(clk), C.byref(mem)), "rt_device_info")
        return {"sm_count": sm.value, "clock_khz": clk.value, "mem_bytes": mem.value}

    # -- scene (main.cu:388-401) --
    def create_world(self, n: int, radius: float = 0.1, precision: int = PREC_FP32):
        self._ck(self.L.rt_scene_generate_ex(self._ctx, n, radius, precision), "rt_scene_generate_ex")
        self.n = n
        return self

    def upload_world(self, spheres: np.ndarray):
        spheres = np.ascontiguousarray(spheres, dtype=SPHERE_DTYPE)
        self._ck(self.L.rt_scene_upload(self._ctx, spheres.ctypes.data, len(spheres)), "rt_scene_upload")
        self.n = len(spheres)
        return self

    def spheres(self) -> np.ndarray:
        out = np.zeros(self.n, dtype=SPHERE_DTYPE)
        self._ck(self.L.rt_scene_download(self._ctx, out.ctypes.data, self.n), "rt_scene_download")
        return out

    def set_camera(self, nx: int, ny: int, desc: CameraDesc | None = None):
        self._ck(self.L.rt_camera_set(self._ctx, C.byref(desc) if desc else None, nx, ny), "rt_camera_set")

    def camera(self) -> np.ndarray:
        out = np.zeros(22, dtype=np.float32)
        self._ck(self.L.rt_camera_get(self._ctx, out.ctypes.data), "rt_camera_get")
        return out

    def camera_half(self, nx: int, ny: int) -> np.ndarray:
        """The camera of the USE_FP16 build for an nx x ny frame (half values widened to float)."""
        out = np.zeros(22, dtype=np.float32)
        self._ck(self.L.rt_camera_get_half(self._ctx, nx, ny, out.ctypes.data), "rt_camera_get_half")
        return out

    # -- octree (main.cu:405-415) --
    def build_octree(self, spheres_per_leaf: int = 30, precision: int = PREC_FP32) -> dict:
        st = OctreeStats()
        self._ck(self.L.rt_octree_build_ex(self._ctx, spheres_per_leaf, precision, C.byref(st)), "rt_octree_build_ex")
        self.spl = spheres_per_leaf
        self.octree_precision = precision
        return st.as_dict()

    def export_octree(self) -> np.ndarray:
        """The tree in the reference's Octree layout; a tree built with PREC_FP16 in the USE_FP16 one (48-byte nodes)."""
        n = self.L.rt_octree_reference_bytes_ex(self.spl, self.octree_precision)
        blob = np.zeros(n, dtype=np.uint8)
        self._ck(self.L.rt_octree_export_reference(self._ctx, blob.ctypes.data, n), "rt_octree_export_reference")
        return blob

    def debug_tree(self) -> dict:
        """Test hook: the internal traversal arrays as raw bytes."""
        names = ["grid", "vox", "refs", "ent_off", "ent_cell", "big_refs", "sph_flag", "cell_start", "cell_list"]
        out = {}
        for k, name in enumerate(names):
            n = self.L.rt_octree_debug_read(self._ctx, k, None, 0)
            buf = np.zeros(max(n, 1), dtype=np.uint8)
            if n:
                got = self.L.rt_octree_debug_read(self._ctx, k, buf.ctypes.data, n)
                assert got == n
            out[name] = buf[:n]
        return out

    def debug_counters(self) -> np.ndarray:
        """Test hook: raw device counters of the last render (see rt_abi.h)."""
        out = np.zeros(32, dtype=np.uint64)
        self._ck(self.L.rt_debug_counters(self._ctx, out.ctypes.data), "rt_debug_counters")
        return out

    def trace_rays(self, origins: np.ndarray, dirs: np.ndarray, use_octree: bool, precision: int = PREC_FP32):
        """Test hook: closest hit per ray -> (idx[n] int32, t[n] float32).  PREC_FP16: the USE_FP16 build's hitTree /
        hitable_list::hit (inputs rounded to half, t a half widened to float, +inf on a miss)."""
        o = np.ascontiguousarray(origins, dtype=np.float32)
        d = np.ascontiguousarray(dirs, dtype=np.float32)
        n = len(o)
        idx = np.zeros(n, dtype=np.int32)
        t = np.zeros(n, dtype=np.float32)
        self._ck(self.L.rt_trace_rays_ex(self._ctx, int(use_octree), precision, n, o.ctypes.data, d.ctypes.data, idx.ctypes.data,
                                         t.ctypes.data), "rt_trace_rays_ex")
        return idx, t

    def camera_rays(self, s: np.ndarray, t: np.ndarray, states: np.ndarray, precision: int = PREC_FP32):
        """camera::get_ray for n (s, t) pairs; `states` [n, 6] uint32 is advanced in place.  Returns (org[n,3], dir[n,3]).
        PREC_FP16: with the USE_FP16 build's camera, s and t rounded to half, rays as halves widened to float."""
        s = np.ascontiguousarray(s, dtype=np.float32); t = np.ascontiguousarray(t, dtype=np.float32)
        assert states.dtype == np.uint32 and states.flags.c_contiguous and states.shape == (len(s), 6)
        org = np.zeros((len(s), 3), np.float32); d = np.zeros((len(s), 3), np.float32)
        self._ck(self.L.rt_camera_get_rays_ex(self._ctx, precision, len(s), s.ctypes.data, t.ctypes.data, states.ctypes.data, org.ctypes.data,
                                              d.ctypes.data), "rt_camera_get_rays_ex")
        return org, d

    def scatter_rays(self, idx: np.ndarray, org: np.ndarray, dirs: np.ndarray, t_hit: np.ndarray, states: np.ndarray,
                     precision: int = PREC_FP32):
        """material::scatter for n hits; returns dict(p, normal, dir, atten, scattered); `states` advanced in place.
        PREC_FP16: the USE_FP16 build's hit record and scatter (inputs rounded to half, outputs halves widened to float)."""
        idx = np.ascontiguousarray(idx, dtype=np.int32); org = np.ascontiguousarray(org, dtype=np.float32)
        dirs = np.ascontiguousarray(dirs, dtype=np.float32); t_hit = np.ascontiguousarray(t_hit, dtype=np.float32)
        n = len(idx)
        assert states.dtype == np.uint32 and states.flags.c_contiguous and states.shape == (n, 6)
        out = {k: np.zeros((n, 3), np.float32) for k in ("p", "normal", "dir", "atten")}
        out["scattered"] = np.zeros(n, np.int32)
        self._ck(self.L.rt_scatter_rays_ex(self._ctx, precision, n, idx.ctypes.data, org.ctypes.data, dirs.ctypes.data, t_hit.ctypes.data,
                                           states.ctypes.data, out["p"].ctypes.data, out["normal"].ctypes.data, out["dir"].ctypes.data,
                                           out["atten"].ctypes.data, out["scattered"].ctypes.data), "rt_scatter_rays_ex")
        return out

    # -- render (main.cu:424-429) --
    @staticmethod
    def args(nx, ny, ns, use_octree, max_depth=50, shard_mode=SHARD_NONE, shard_rank=0, shard_count=1,
             seed_mode=SEED_HEAD, precision=PREC_FP32, variant=0) -> RenderArgs:
        a = RenderArgs(nx, ny, ns, max_depth, int(bool(use_octree)), seed_mode, shard_mode, shard_rank, shard_count, precision)
        a.tune[1] = variant          # kernel variant for A/B runs and tests (0 = automatic); it never changes the image
        return a

    def render(self, nx, ny, ns, use_octree=True, **kw):
        """Whole frame with a HOST destination (render + device->host copy).  Returns (fb[ny,nx,3], stats)."""
        a = self.args(nx, ny, ns, use_octree, **kw)
        fb = np.empty((ny, nx, 3), dtype=np.float32)
        st = RenderStats()
        self._ck(self.L.rt_render_to_host(self._ctx, C.byref(a), fb.ctypes.data, C.byref(st)), "rt_render_to_host")
        return fb, st.as_dict()

    def render_pixels(self, nx, ny, ns, pixels, use_octree=True, finalize=True, **kw):
        """The listed pixels (host array of indices j*nx + i, any order, duplicates allowed) of the nx x ny frame, exactly as
        render() (finalize) or render_accumulate() (linear sums) computes them.  Returns (values[count, 3] float32, stats);
        an index >= nx*ny comes back as (0, 0, 0).  window_pixels() lists a rectangle."""
        import torch
        pix = np.ascontiguousarray(pixels, dtype=np.uint32).reshape(-1)
        dev = torch.device("cuda", self.device)
        pix_dev = torch.from_numpy(pix.view(np.int32)).to(dev)          # the same 32-bit patterns
        out = torch.empty((len(pix), 3), dtype=torch.float32, device=dev)
        st = self.render_pixels_device(self.args(nx, ny, ns, use_octree, **kw), pix_dev.data_ptr(), len(pix), out.data_ptr(), finalize)
        return out.cpu().numpy(), st

    def render_pixels_device(self, args: RenderArgs, pixels_ptr: int, count: int, out_ptr: int, finalize=True, want_stats=True):
        """rt_render_pixels on device pointers: `count` uint32 pixel indices at pixels_ptr, count*3 floats to out_ptr (list order).
        want_stats=False keeps the call asynchronous (last_render_stats() reads them later)."""
        st = RenderStats()
        self._ck(self.L.rt_render_pixels(self._ctx, C.byref(args), C.c_void_p(pixels_ptr), count, C.c_void_p(out_ptr), int(bool(finalize)),
                                         C.byref(st) if want_stats else None), "rt_render_pixels")
        return st.as_dict() if want_stats else None

    def format_ppm_device(self, fb_dev_ptr: int, nx: int, ny: int) -> bytes:
        """output_to_stream (main.cu:321-333) on the device: P3 text of a DEVICE frame; only the text is copied back."""
        n = C.c_size_t()
        self._ck(self.L.rt_ppm_format(self._ctx, C.c_void_p(fb_dev_ptr), nx, ny, C.byref(n)), "rt_ppm_format")
        buf = C.create_string_buffer(max(n.value, 1))
        self._ck(self.L.rt_ppm_read(self._ctx, buf, n.value), "rt_ppm_read")
        return buf.raw[:n.value]

    def render_ppm(self, nx, ny, ns, use_octree=True, **kw):
        """render + output_to_stream without the float frame ever leaving the GPU.  Returns (P3 text, stats)."""
        a = self.args(nx, ny, ns, use_octree, **kw)
        st, n = RenderStats(), C.c_size_t()
        self._ck(self.L.rt_render_to_ppm(self._ctx, C.byref(a), C.byref(st), C.byref(n)), "rt_render_to_ppm")
        buf = C.create_string_buffer(max(n.value, 1))
        self._ck(self.L.rt_ppm_read(self._ctx, buf, n.value), "rt_ppm_read")
        return buf.raw[:n.value], st.as_dict()

    def render_device(self, args: RenderArgs, fb_dev_ptr: int, want_stats=True):
        st = RenderStats()
        self._ck(self.L.rt_render(self._ctx, C.byref(args), C.c_void_p(fb_dev_ptr), C.byref(st) if want_stats else None),
                 "rt_render")
        return st.as_dict() if want_stats else None

    def render_accumulate(self, args: RenderArgs, accum_dev_ptr: int, want_stats=True):
        st = RenderStats()
        self._ck(self.L.rt_render_accumulate(self._ctx, C.byref(args), C.c_void_p(accum_dev_ptr),
                                             C.byref(st) if want_stats else None), "rt_render_accumulate")
        return st.as_dict() if want_stats else None

    def render_progressive(self, args: RenderArgs, accum_dev_ptr: int, state_dev_ptr: int, first: bool, want_stats=True):
        """args.ns MORE samples per pixel, continuing every pixel's stream and sum (render_progressive, main.cu:119-142)."""
        st = RenderStats()
        self._ck(self.L.rt_render_progressive(self._ctx, C.byref(args), C.c_void_p(accum_dev_ptr), C.c_void_p(state_dev_ptr), int(first),
                                              C.byref(st) if want_stats else None), "rt_render_progressive")
        return st.as_dict() if want_stats else None

    def last_render_stats(self) -> dict:
        """Statistics of the last render call made with want_stats=False (waits for the stream)."""
        st = RenderStats()
        self._ck(self.L.rt_last_render_stats(self._ctx, C.byref(st)), "rt_last_render_stats")
        return st.as_dict()

    def finalize(self, accum_dev_ptr: int, fb_dev_ptr: int, nx, ny, ns):
        self._ck(self.L.rt_finalize(self._ctx, C.c_void_p(accum_dev_ptr), C.c_void_p(fb_dev_ptr), nx, ny, ns), "rt_finalize")

    def finalize_n(self, accum_dev_ptr: int, fb_dev_ptr: int, count: int, ns: int):
        self._ck(self.L.rt_finalize_n(self._ctx, C.c_void_p(accum_dev_ptr), C.c_void_p(fb_dev_ptr), count, ns), "rt_finalize_n")

    def finalize_ex(self, accum_dev_ptr: int, fb_dev_ptr: int, count: int, ns: int, precision: int):
        """/ns and sqrt on `count` linear sums in the given arithmetic (PREC_FP16: the sums are halves widened to float)."""
        self._ck(self.L.rt_finalize_ex(self._ctx, C.c_void_p(accum_dev_ptr), C.c_void_p(fb_dev_ptr), count, ns, precision),
                 "rt_finalize_ex")

    def hfma2_peak_tflops(self) -> float:
        """Measured dense packed-half HFMA2 rate (TFLOP/s, 4 flop per instruction): the USE_FP16 roofline denominator."""
        t, ms = C.c_float(), C.c_float()
        self._ck(self.L.rt_hfma2_peak(self._ctx, C.byref(t), C.byref(ms)), "rt_hfma2_peak")
        return float(t.value)

    def ffma_peak_tflops(self) -> float:
        """Measured dense FP32 FFMA rate (TFLOP/s) of this GPU: the FP32 roofline denominator."""
        t, ms = C.c_float(), C.c_float()
        self._ck(self.L.rt_ffma_peak(self._ctx, C.byref(t), C.byref(ms)), "rt_ffma_peak")
        return float(t.value)

    def synchronize(self):
        self._ck(self.L.rt_synchronize(self._ctx), "rt_synchronize")
