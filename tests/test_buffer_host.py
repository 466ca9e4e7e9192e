"""CPU tier of the library's scratch buffers: csrc/rt_buffer.h compiled for the host against a shim of cudaMalloc / cudaFree /
cudaMallocHost / cudaFreeHost (malloc-backed, counting live blocks of each kind, with one chosen allocation call made to fail).
No CUDA runtime is linked: the shim is the only allocator the header sees."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "dd2360-raytracing_b200", "csrc")
CUDA_ERROR_MEMORY_ALLOCATION = 2           # cudaErrorMemoryAllocation

SHIM = r"""
#include <stdlib.h>
#include <map>
#include "rt_buffer.h"

namespace {
enum Kind { kDevice = 0, kPinned = 1 };
std::map<void *, Kind> live;
int calls = 0, fail_on = -1, bad_frees = 0;
size_t last_bytes = 0;
cudaError_t alloc(void **p, size_t bytes, Kind k) {
    if (calls++ == fail_on) {
        *p = reinterpret_cast<void *>(0x10);  // what a failed call leaves in *p is not promised: the buffer must not keep it
        return cudaErrorMemoryAllocation;
    }
    *p = malloc(bytes);
    live[*p] = k;
    last_bytes = bytes;
    return cudaSuccess;
}
cudaError_t release(void *p, Kind k) {
    auto it = live.find(p);
    if (it == live.end() || it->second != k) {
        bad_frees++;
        return cudaErrorInvalidValue;
    }
    live.erase(it);
    free(p);
    return cudaSuccess;
}
}  // namespace

extern "C" {
cudaError_t cudaMalloc(void **p, size_t bytes) { return alloc(p, bytes, kDevice); }
cudaError_t cudaMallocHost(void **p, size_t bytes) { return alloc(p, bytes, kPinned); }
cudaError_t cudaFree(void *p) { return release(p, kDevice); }
cudaError_t cudaFreeHost(void *p) { return release(p, kPinned); }

int live_blocks(int kind) {
    int n = 0;
    for (const auto &b : live) n += b.second == kind;
    return n;
}
int alloc_calls() { return calls; }
int bad_free_calls() { return bad_frees; }
size_t last_alloc_bytes() { return last_bytes; }
void fail_call(int k) { fail_on = k; }       // the allocation call with this number fails (alloc_calls() is the next one)
}

#define BUFFER_API(name, Type)                                                                     \
    extern "C" void *name##_new() { return new Type; }                                             \
    extern "C" void name##_delete(void *b) { delete static_cast<Type *>(b); }                      \
    extern "C" int name##_reserve(void *b, size_t need, size_t slack) { return static_cast<Type *>(b)->reserve(need, slack); } \
    extern "C" void *name##_ptr(void *b) { return static_cast<Type *>(b)->ptr; }                   \
    extern "C" size_t name##_cap(void *b) { return static_cast<Type *>(b)->cap; }
using Device = rt::Buffer<double>;
using Pinned = rt::Buffer<double, rt::Mem::Pinned>;
BUFFER_API(dev, Device)
BUFFER_API(pin, Pinned)
"""

DEVICE, PINNED = 0, 1


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("buffer_shim")
    src, so = d / "shim.cpp", d / "libbuffer_shim.so"
    src.write_text(SHIM)
    # -Bsymbolic: the header's calls bind to the shim's allocator even when a CUDA runtime is already loaded in the process (torch's)
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Werror", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-I", CSRC, "-I/usr/local/cuda/include",
                    str(src), "-o", str(so)], check=True)
    L = C.CDLL(str(so))
    L.last_alloc_bytes.restype = C.c_size_t
    for kind in ("dev", "pin"):
        getattr(L, f"{kind}_new").restype = C.c_void_p
        getattr(L, f"{kind}_delete").argtypes = [C.c_void_p]
        getattr(L, f"{kind}_reserve").argtypes = [C.c_void_p, C.c_size_t, C.c_size_t]
        getattr(L, f"{kind}_ptr").restype = C.c_void_p
        getattr(L, f"{kind}_ptr").argtypes = [C.c_void_p]
        getattr(L, f"{kind}_cap").restype = C.c_size_t
        getattr(L, f"{kind}_cap").argtypes = [C.c_void_p]
    return L


class Buf:
    """One Buffer<double> (kind "dev") or Buffer<double, Mem::Pinned> (kind "pin") of the shim."""

    def __init__(self, L, kind):
        self.L, self.kind = L, kind
        self.h = getattr(L, f"{kind}_new")()

    def reserve(self, need, slack=0):
        return getattr(self.L, f"{self.kind}_reserve")(self.h, need, slack)

    @property
    def ptr(self):
        return getattr(self.L, f"{self.kind}_ptr")(self.h)

    @property
    def cap(self):
        return getattr(self.L, f"{self.kind}_cap")(self.h)

    def delete(self):
        getattr(self.L, f"{self.kind}_delete")(self.h)


@pytest.fixture
def L(shim):
    yield shim
    assert shim.live_blocks(DEVICE) == 0 and shim.live_blocks(PINNED) == 0
    assert shim.bad_free_calls() == 0


@pytest.mark.parametrize("kind", ["dev", "pin"])
def test_failed_reserve_leaves_buffer_empty_and_next_reserve_allocates(L, kind):
    live_kind = DEVICE if kind == "dev" else PINNED
    b = Buf(L, kind)
    L.fail_call(L.alloc_calls())                           # the very first allocation fails
    assert b.reserve(8) == CUDA_ERROR_MEMORY_ALLOCATION
    assert (b.ptr, b.cap) == (None, 0)
    assert b.reserve(8) == 0 and b.ptr is not None and b.cap == 8
    L.fail_call(L.alloc_calls())                           # a growth that fails releases the old block and keeps nothing
    assert b.reserve(100, 10) == CUDA_ERROR_MEMORY_ALLOCATION
    assert (b.ptr, b.cap) == (None, 0)
    assert L.live_blocks(live_kind) == 0
    assert b.reserve(4) == 0 and b.cap == 4                # and the next call tries again, at the size it asks for
    assert L.live_blocks(live_kind) == 1
    b.delete()


def test_reserve_within_capacity_allocates_nothing(L):
    b = Buf(L, "dev")
    assert b.reserve(10, 5) == 0
    calls, ptr = L.alloc_calls(), b.ptr
    for need in (0, 1, 10, 15):
        assert b.reserve(need) == 0 and b.reserve(need, 1000) == 0
    assert L.alloc_calls() == calls and b.ptr == ptr and b.cap == 15
    assert b.reserve(16) == 0 and L.alloc_calls() == calls + 1 and b.cap == 16
    b.delete()


def test_reserve_allocates_need_plus_slack_elements(L):
    b = Buf(L, "dev")
    assert b.reserve(10, 5) == 0 and b.cap == 15 and L.last_alloc_bytes() == 15 * 8
    assert b.reserve(16, 4) == 0 and b.cap == 20 and L.last_alloc_bytes() == 20 * 8
    assert b.reserve(21) == 0 and b.cap == 21 and L.last_alloc_bytes() == 21 * 8
    b.delete()


def test_device_and_pinned_buffers_release_through_their_own_free(L):
    d, p = Buf(L, "dev"), Buf(L, "pin")
    assert d.reserve(3) == 0 and p.reserve(3) == 0
    assert L.live_blocks(DEVICE) == 1 and L.live_blocks(PINNED) == 1
    assert d.reserve(30) == 0 and p.reserve(30) == 0      # growth frees the old block of each kind
    assert L.live_blocks(DEVICE) == 1 and L.live_blocks(PINNED) == 1
    d.delete()
    assert L.live_blocks(DEVICE) == 0 and L.live_blocks(PINNED) == 1
    p.delete()
    assert L.bad_free_calls() == 0


def test_no_block_live_after_the_buffers_are_destroyed(L):
    bufs = [Buf(L, kind) for kind in ("dev", "pin") * 4]
    for i, b in enumerate(bufs):
        if i % 3 == 0:
            L.fail_call(L.alloc_calls())
        b.reserve(1 + i, i)
        b.reserve(20 + i)
    assert L.live_blocks(DEVICE) + L.live_blocks(PINNED) == len(bufs)
    never = Buf(L, "dev")                                  # a buffer that never allocated frees nothing
    for b in bufs + [never]:
        b.delete()
    assert L.live_blocks(DEVICE) == 0 and L.live_blocks(PINNED) == 0
