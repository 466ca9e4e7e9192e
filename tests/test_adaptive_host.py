"""CPU tier of rt_render_adaptive: the noise estimate e_p (csrc/rt_adaptive.h) compiled for the host and compared bit for bit with
a numpy restatement over about a million inputs, and the parts of the Python binding that need no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dd2360-raytracing_b200", "csrc")

SHIM = r"""
#include "rt_adaptive.h"
extern "C" void adaptive_errors(const float *s, const uint32_t *a, const float *x, const uint32_t *c, float *out, size_t n) {
    for (size_t i = 0; i < n; i++) out[i] = rt::adaptive_error(s + 3 * i, a[i], x + 3 * i, c[i]);
}
"""


@pytest.fixture(scope="module")
def metric(tmp_path_factory):
    d = tmp_path_factory.mktemp("adaptive_metric")
    src, so = d / "shim.cpp", d / "libadaptive_metric.so"
    src.write_text(SHIM)
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    L = C.CDLL(str(so))
    L.adaptive_errors.restype = None
    L.adaptive_errors.argtypes = [C.c_void_p] * 5 + [C.c_size_t]

    def run(s, a, x, c):
        s, x = np.ascontiguousarray(s, np.float32), np.ascontiguousarray(x, np.float32)
        a, c = np.ascontiguousarray(a, np.uint32), np.ascontiguousarray(c, np.uint32)
        out = np.empty(len(a), np.float32)
        L.adaptive_errors(s.ctypes.data, a.ctypes.data, x.ctypes.data, c.ctypes.data, out.ctypes.data, len(a))
        return out
    return run


def metric_model(s, a, x, c):
    """e_p as the issue of the feature defines it, in float32 numpy (every operation rounded once, IEEE)."""
    f32 = np.float32
    fa, fb, fc = a.astype(f32), (c - a).astype(f32), c.astype(f32)
    with np.errstate(all="ignore"):
        A = s / fa[:, None]
        B = (x - s) / fb[:, None]
        dk = np.abs(np.sqrt(A) - np.sqrt(B))
        d = np.maximum(np.maximum(dk[:, 0], dk[:, 1]), dk[:, 2])
        w = (np.sqrt(fa) * np.sqrt(fb)) / fc
        return d * w


def _same(got, want):
    gb, wb = got.view(np.uint32), want.view(np.uint32)
    nan = np.isnan(want)
    return bool((np.isnan(got) == nan).all() and (gb[~nan] == wb[~nan]).all())


def _inputs(n, seed):
    rng = np.random.default_rng(seed)
    groups = []
    m = n // 8
    # realistic: radiance sums of a >= 1 and b >= 1 samples, counts up to the 65536 budget
    a = rng.integers(1, 32768, m).astype(np.uint32)
    b = rng.integers(1, 32768, m).astype(np.uint32)
    mean = rng.random((m, 3), dtype=np.float32) * 4
    s = (mean * a[:, None] * rng.uniform(0.5, 1.5, (m, 3))).astype(np.float32)
    x = (s + mean * b[:, None] * rng.uniform(0.5, 1.5, (m, 3))).astype(np.float32)
    groups.append((s, a, x, a + b))
    # a = b (the first estimate: two segments of min_spp/2), and small counts
    a = rng.integers(1, 65, m).astype(np.uint32)
    s = (rng.random((m, 3), dtype=np.float32) * a[:, None]).astype(np.float32)
    x = (s + rng.random((m, 3), dtype=np.float32) * a[:, None]).astype(np.float32)
    groups.append((s, a, x, 2 * a))
    # unequal segments: doubling rounds and a capped last round
    a = (2 ** rng.integers(1, 15, m)).astype(np.uint32)
    b = np.where(rng.random(m) < 0.5, a, rng.integers(1, 65536, m).astype(np.uint32) % a + 1).astype(np.uint32)
    s = (rng.random((m, 3), dtype=np.float32) * a[:, None]).astype(np.float32)
    x = (s + rng.random((m, 3), dtype=np.float32) * b[:, None]).astype(np.float32)
    groups.append((s, a, x, a + b))
    # zero sums (sky-free black pixels), and x == s (an empty second segment's worth of light)
    a = rng.integers(1, 1000, m).astype(np.uint32)
    z = np.zeros((m, 3), np.float32)
    s = np.where(rng.random((m, 1)) < 0.5, z, rng.random((m, 3), dtype=np.float32)).astype(np.float32)
    x = np.where(rng.random((m, 1)) < 0.5, s, s * 2).astype(np.float32)
    groups.append((s, a, x, a + rng.integers(1, 1000, m).astype(np.uint32)))
    # denormals
    a = rng.integers(1, 64, m).astype(np.uint32)
    s = rng.integers(1, 1 << 23, (m, 3)).astype(np.uint32).view(np.float32)
    x = (s + rng.integers(0, 1 << 22, (m, 3)).astype(np.uint32).view(np.float32)).astype(np.float32)
    groups.append((s, a, x, a + rng.integers(1, 64, m).astype(np.uint32)))
    # arbitrary bit patterns (negative, huge, inf, NaN included)
    a = rng.integers(1, 65536, m).astype(np.uint32)
    s = rng.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32).view(np.float32)
    x = rng.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32).view(np.float32)
    groups.append((s, a, x, a + rng.integers(1, 65536, m).astype(np.uint32)))
    # inf and NaN in one channel of otherwise ordinary sums
    a = rng.integers(1, 256, 2 * m).astype(np.uint32)
    s = (rng.random((2 * m, 3), dtype=np.float32) * a[:, None]).astype(np.float32)
    x = (s * 2).astype(np.float32)
    ch = rng.integers(0, 3, 2 * m)
    bad = rng.choice(np.array([np.inf, np.nan, -np.inf], np.float32), 2 * m)
    which = rng.integers(0, 3, 2 * m)                  # 0: in x, 1: in s, 2: in both
    rows = np.arange(2 * m)
    x[rows[which != 1], ch[which != 1]] = bad[which != 1]
    s[rows[which != 0], ch[which != 0]] = bad[which != 0]
    groups.append((s, a, x, 2 * a))
    return [np.concatenate(g) for g in zip(*groups)]


def test_metric_matches_numpy_restatement(metric):
    s, a, x, c = _inputs(1 << 20, 1)
    assert len(a) >= 1_000_000
    got = metric(s, a, x, c)
    want = metric_model(s, a, x, c)
    assert _same(got, want)
    assert np.isnan(want).any() and np.isinf(want).any() and (want == 0).any()
    assert ((s != 0) & (np.abs(s) < np.finfo(np.float32).tiny)).any()        # denormal sums are among the inputs


def test_metric_edge_cases(metric):
    f = np.float32
    s = np.array([[0, 0, 0], [1, 2, 3], [1, 1, 1], [1, 1, 1], [1, 1, 1], [np.inf, 1, 1], [np.nan, 1, 1], [1, 1, 1]], f)
    x = np.array([[0, 0, 0], [2, 4, 6], [3, 2, 2], [np.inf, 2, 2], [np.nan, 2, 2], [np.inf, 2, 2], [np.nan, 2, 2], [1, 1, 1]], f)
    a = np.array([4, 8, 1, 2, 2, 2, 2, 8], np.uint32)
    c = np.array([8, 16, 2, 4, 4, 4, 4, 16], np.uint32)
    got = metric(s, a, x, c)
    assert _same(got, metric_model(s, a, x, c))
    assert got[0] == 0 and got[1] == 0                      # no light, and two segments with the same mean: converged
    assert got[2] > 0 and got[7] > 0                        # an empty second segment differs from a lit first one
    # a non-finite sum never counts as converged: the tile rule !(E_t <= threshold) refines it at any finite threshold
    for k in (3, 4, 5, 6):
        assert not (got[k] <= f(3e38)), (k, got[k])


def test_binding_structs_and_symbols(pkg):
    assert C.sizeof(pkg.AdaptiveParams) == 32
    assert C.sizeof(pkg.AdaptiveStats) == 184
    assert C.sizeof(pkg.RenderStats) == 48 and pkg.AdaptiveStats.round_pixels.offset == 56
    assert "rt_render_adaptive" in pkg.ABI_SYMBOLS
    L = pkg.load_library()
    fn = L.rt_render_adaptive
    vp = C.c_void_p
    assert fn.restype is C.c_int
    assert fn.argtypes == [vp, C.POINTER(pkg.RenderArgs), C.POINTER(pkg.AdaptiveParams), vp, vp, vp, vp, vp, C.POINTER(pkg.AdaptiveStats)]
    p = pkg.AdaptiveParams(8, float("inf"))
    assert p.min_spp == 8 and p.threshold == float("inf") and list(p.reserved) == [0] * 6
