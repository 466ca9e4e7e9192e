"""ctypes bindings for the CPU ORACLE (test infrastructure, NOT product code).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this module.
It wraps oracle/librt_oracle.so (the plain-C restatement, rt_oracle.h) and, when present, the reference-backed
checkers under oracle/_ref/ (libref_host_*.so: the reference's own headers compiled for the host).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

SPHERE_DTYPE = np.dtype(
    [("cx", "<f4"), ("cy", "<f4"), ("cz", "<f4"), ("radius", "<f4"), ("mat", "<i4"),
     ("ax", "<f4"), ("ay", "<f4"), ("az", "<f4"), ("param", "<f4")]
)
assert SPHERE_DTYPE.itemsize == 36

ARITH_HOST, ARITH_DEVICE = 0, 1
NUMBER_NODES, NUMBER_LEAFS, NODE_INTS = 585, 4096, 15


class Camera(C.Structure):
    _fields_ = [(n, C.c_float * 3) for n in ("origin", "lower_left_corner", "horizontal", "vertical", "u", "v", "w")] + [
        ("lens_radius", C.c_float)]

    def as_array(self) -> np.ndarray:
        return np.frombuffer(bytes(self), dtype="<f4").copy()


class Counters(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("sphere_tests", C.c_uint64), ("aabb_tests", C.c_uint64),
                ("paths", C.c_uint64), ("max_depth", C.c_uint32)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class OctreeStats(C.Structure):
    _fields_ = [("node_count", C.c_int32), ("leaf_count", C.c_int32), ("entries", C.c_int64),
                ("dropped_full", C.c_int64), ("dropped_outside", C.c_int64)]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class RenderParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("nx", "ny", "ns", "use_octree", "spl", "arith", "seed_mode", "max_depth",
                                       "i0", "i1", "istep", "j0", "j1", "jstep", "threads")]


SEED_HEAD, SEED_UPSTREAM = 0, 1


def make_params(nx, ny, ns, use_octree, spl=30, arith=ARITH_DEVICE, window=None, step=(1, 1), threads=0,
                max_depth=50, seed_mode=SEED_HEAD) -> RenderParams:
    i0, i1, j0, j1 = window if window else (0, nx, 0, ny)
    return RenderParams(nx, ny, ns, int(use_octree), spl, arith, seed_mode, max_depth, i0, i1, step[0], j0, j1, step[1], threads)


def build(force: bool = False) -> str:
    """Compile the C restatement (gcc; seconds).  Building the checker is not using it."""
    so = os.path.join(HERE, "librt_oracle.so")
    srcs = [os.path.join(HERE, f) for f in ("rt_oracle.c", "rt_oracle_core.inc.h", "rt_oracle.h")]
    if force or not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        env = {k: v for k, v in os.environ.items() if k not in ("CC", "CXX")}
        subprocess.run(["make", "-C", HERE, "oracle"], check=True, env=env, capture_output=True)
    return so


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.rto_create_world.restype = C.c_int
        L.rto_create_world.argtypes = [C.c_int, C.c_float, C.c_void_p]
        L.rto_camera_init.argtypes = [C.POINTER(Camera), C.c_int, C.c_int, C.c_int]
        L.rto_octree_sizeof.restype = C.c_size_t
        L.rto_octree_sizeof.argtypes = [C.c_int]
        L.rto_build_octree.restype = C.c_int
        L.rto_build_octree.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(OctreeStats)]
        L.rto_render.restype = C.c_int
        L.rto_render.argtypes = [C.c_void_p, C.c_int, C.POINTER(Camera), C.c_void_p, C.POINTER(RenderParams),
                                 C.c_void_p, C.c_void_p, C.POINTER(Counters)]
        L.rto_quantise.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        L.rto_write_ppm.restype = C.c_size_t
        L.rto_write_ppm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t]
        L.rto_xorwow_stream.argtypes = [C.c_uint64, C.c_int, C.c_void_p, C.c_void_p]
        L.rto_xorwow_state.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
        L.rto_xorwow_skip_tables.argtypes = [C.c_void_p, C.c_int]
        L.rto_closest_hit.restype = C.c_int
        L.rto_closest_hit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        L.rto_closest_hits.restype = None
        L.rto_closest_hits.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.rto_version.restype = C.c_char_p
        _lib = L
    return _lib


def _p(a: np.ndarray | None):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def create_world(n: int, radius: float = 0.1):
    out = np.zeros(n, dtype=SPHERE_DTYPE)
    written = lib().rto_create_world(n, radius, _p(out))
    return out, written


def camera(nx: int, ny: int, arith: int = ARITH_DEVICE) -> Camera:
    cam = Camera()
    lib().rto_camera_init(C.byref(cam), nx, ny, arith)
    return cam


def octree_sizeof(spl: int) -> int:
    return int(lib().rto_octree_sizeof(spl))


def build_octree(spheres: np.ndarray, spl: int):
    blob = np.zeros(octree_sizeof(spl), dtype=np.uint8)
    st = OctreeStats()
    lib().rto_build_octree(_p(spheres), len(spheres), spl, _p(blob), C.byref(st))
    return blob, st.as_dict()


def split_octree(blob: np.ndarray, spl: int):
    """View a reference-layout Octree blob as (nodes[585,15] int32, leaves[4097,spl+1] int32, nodeCount, leafCount)."""
    ints = blob.view("<i4")
    nn = NUMBER_NODES * NODE_INTS
    nl = (NUMBER_LEAFS + 1) * (spl + 1)
    nodes = ints[:nn].reshape(NUMBER_NODES, NODE_INTS)
    leaves = ints[nn:nn + nl].reshape(NUMBER_LEAFS + 1, spl + 1)
    return nodes, leaves, int(ints[nn + nl]), int(ints[nn + nl + 1])


def render(spheres, cam: Camera, params: RenderParams, blob=None, want_linear=False):
    nx, ny = params.nx, params.ny
    fb = np.zeros((ny, nx, 3), dtype=np.float32)
    lin = np.zeros((ny, nx, 3), dtype=np.float32) if want_linear else None
    ctr = Counters()
    rc = lib().rto_render(_p(spheres), len(spheres), C.byref(cam), _p(blob), C.byref(params), _p(fb), _p(lin), C.byref(ctr))
    if rc != 0:
        raise RuntimeError(f"rto_render failed: {rc}")
    return fb, lin, ctr.as_dict()


def quantise(fb: np.ndarray) -> np.ndarray:
    ny, nx, _ = fb.shape
    out = np.zeros((ny, nx, 3), dtype=np.uint8)
    lib().rto_quantise(_p(np.ascontiguousarray(fb)), nx, ny, _p(out))
    return out


def write_ppm(fb: np.ndarray) -> bytes:
    ny, nx, _ = fb.shape
    fb = np.ascontiguousarray(fb, dtype=np.float32)
    need = lib().rto_write_ppm(_p(fb), nx, ny, None, 0)
    buf = C.create_string_buffer(need)
    lib().rto_write_ppm(_p(fb), nx, ny, buf, need)
    return buf.raw[:need]


def xorwow_stream(seed: int, count: int):
    u = np.zeros(count, dtype=np.uint32)
    f = np.zeros(count, dtype=np.float32)
    lib().rto_xorwow_stream(seed, count, _p(u), _p(f))
    return u, f


def xorwow_state(seed: int, subsequence: int) -> np.ndarray:
    """{d, v0..v4} after curand_init(seed, subsequence, 0), from the restatement."""
    out = np.zeros(6, dtype=np.uint32)
    lib().rto_xorwow_state(C.c_uint64(seed), C.c_uint64(subsequence), _p(out))
    return out


def xorwow_skip_tables(bits: int = 40) -> np.ndarray:
    """The GF(2) skip matrices T^(2^(67+k)): [bits, 160, 5] uint32."""
    out = np.zeros((bits, 160, 5), dtype=np.uint32)
    n = lib().rto_xorwow_skip_tables(_p(out), bits)
    return out[:n]


def closest_hit(spheres, o, d, blob=None, spl=30, use_octree=False, arith=ARITH_DEVICE):
    o = np.asarray(o, dtype=np.float32)
    d = np.asarray(d, dtype=np.float32)
    t = C.c_float(0)
    idx = lib().rto_closest_hit(_p(spheres), len(spheres), _p(blob), spl, int(use_octree), arith, _p(o), _p(d), C.byref(t))
    return idx, t.value


def closest_hits(spheres, org, dirs, blob=None, spl=30, use_octree=False, arith=ARITH_DEVICE):
    """closest_hit for every row of org / dirs ([R, 3]), OpenMP over the rays: (index int32[R], t float32[R])."""
    org = np.ascontiguousarray(org, dtype=np.float32).reshape(-1, 3)
    dirs = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
    assert org.shape == dirs.shape
    idx = np.zeros(len(org), np.int32)
    t = np.zeros(len(org), np.float32)
    lib().rto_closest_hits(_p(spheres), len(spheres), _p(blob), spl, int(use_octree), arith, len(org), _p(org), _p(dirs),
                           _p(idx), _p(t))
    return idx, t


# ---------------------------------------------------------------------------------------------------------
# reference-backed host checker (oracle/_ref/libref_host_<oct|brute>_spl<SPL>.so), when it has been built
# ---------------------------------------------------------------------------------------------------------
class RefHost:
    def __init__(self, variant: str):
        path = os.path.join(HERE, "_ref", f"libref_host_{variant}.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        L = C.CDLL(path)
        L.refh_create_world.restype = C.c_void_p
        L.refh_create_world.argtypes = [C.c_int, C.c_float, C.c_int, C.c_int]
        L.refh_initialised.argtypes = [C.c_void_p]
        L.refh_export_spheres.argtypes = [C.c_void_p, C.c_void_p]
        L.refh_export_camera.argtypes = [C.c_void_p, C.c_void_p]
        L.refh_octree_sizeof.restype = C.c_size_t
        L.refh_build_octree.argtypes = [C.c_void_p, C.c_void_p]
        L.refh_render.argtypes = [C.c_void_p, C.POINTER(RenderParams), C.c_void_p, C.c_void_p, C.POINTER(Counters)]
        L.refh_closest_hit.restype = C.c_int
        L.refh_closest_hit.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        L.refh_destroy.argtypes = [C.c_void_p]
        if hasattr(L, "refh_curand_state"):
            L.refh_curand_state.argtypes = [C.c_uint64, C.c_uint64, C.c_void_p]
        self.L = L
        self.spl = L.refh_spl()
        self.use_octree = bool(L.refh_use_octree())
        self.world = None

    @staticmethod
    def available(variant: str) -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", f"libref_host_{variant}.so"))

    def create_world(self, n, radius, nx, ny):
        self.destroy()
        self.n = n
        self.world = self.L.refh_create_world(n, radius, nx, ny)
        return self

    def spheres(self):
        out = np.zeros(self.n, dtype=SPHERE_DTYPE)
        self.L.refh_export_spheres(self.world, _p(out))
        return out

    def camera(self):
        out = np.zeros(22, dtype=np.float32)
        self.L.refh_export_camera(self.world, _p(out))
        return out

    def build_octree(self):
        blob = np.zeros(self.L.refh_octree_sizeof(), dtype=np.uint8)
        self.L.refh_build_octree(self.world, _p(blob))
        return blob

    def render(self, params: RenderParams, want_linear=False):
        fb = np.zeros((params.ny, params.nx, 3), dtype=np.float32)
        lin = np.zeros((params.ny, params.nx, 3), dtype=np.float32) if want_linear else None
        ctr = Counters()
        self.L.refh_render(self.world, C.byref(params), _p(fb), _p(lin), C.byref(ctr))
        return fb, lin, ctr.as_dict()

    def curand_state(self, seed: int, subsequence: int) -> np.ndarray:
        """cuRAND's own curand_init(seed, subsequence, 0) (toolkit header compiled for the host)."""
        out = np.zeros(6, dtype=np.uint32)
        self.L.refh_curand_state(seed, subsequence, _p(out))
        return out

    def closest_hit(self, o, d):
        o = np.asarray(o, dtype=np.float32)
        d = np.asarray(d, dtype=np.float32)
        t = C.c_float(0)
        idx = self.L.refh_closest_hit(self.world, _p(o), _p(d), C.byref(t))
        return idx, t.value

    def destroy(self):
        if self.world:
            self.L.refh_destroy(self.world)
            self.world = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass
