// rt_math.cuh — explicitly rounded float arithmetic for the parity-critical math.
//
// The reference is compiled with nvcc's default -fmad=true and ptxas fuses every add/sub that has a product
// operand (read off the SASS of main.cu built for sm_100; the rule is in DESIGN.md §4).  To produce the same
// bits no matter how THIS code is inlined or scheduled, every parity-critical expression is written with
// explicitly rounded primitives that the compiler never re-associates or contracts:
//   device: __fmaf_rn / __fmul_rn / __fadd_rn / __fsub_rn / __fdiv_rn / __fsqrt_rn
//   host  : fmaf / * / + / - / / / sqrtf   (tests/hostsim only; compiled with -ffp-contract=off)
// Code that is NOT parity-critical (pruning, DDA stepping) uses ordinary operators.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define RT_HD __host__ __device__ __forceinline__
#else
#define RT_HD inline
#endif

namespace rt {

#if defined(__CUDA_ARCH__)
RT_HD float fma_(float a, float b, float c) { return __fmaf_rn(a, b, c); }
RT_HD float mul_(float a, float b) { return __fmul_rn(a, b); }
RT_HD float add_(float a, float b) { return __fadd_rn(a, b); }
RT_HD float sub_(float a, float b) { return __fsub_rn(a, b); }
RT_HD float div_(float a, float b) { return __fdiv_rn(a, b); }
RT_HD float sqrt_(float a) { return __fsqrt_rn(a); }
#else
RT_HD float fma_(float a, float b, float c) { return fmaf(a, b, c); }
RT_HD float mul_(float a, float b) { return a * b; }
RT_HD float add_(float a, float b) { return a + b; }
RT_HD float sub_(float a, float b) { return a - b; }
RT_HD float div_(float a, float b) { return a / b; }
RT_HD float sqrt_(float a) { return sqrtf(a); }
#endif

RT_HD int imin(int a, int b) { return a < b ? a : b; }
RT_HD int imax(int a, int b) { return a > b ? a : b; }

struct vec3f {
    float x, y, z;
};
RT_HD vec3f mk(float x, float y, float z) {
    vec3f v;
    v.x = x; v.y = y; v.z = z;
    return v;
}

// vec3.h:91-93 dot(): x1*x2 + y1*y2 + z1*z2 as ptxas fuses it
RT_HD float dot3(vec3f a, vec3f b) { return fma_(a.z, b.z, fma_(a.x, b.x, mul_(a.y, b.y))); }
// vec3.h:146-148 unit_vector(): three true divides by length() (vec3.h:34)
RT_HD vec3f unit_vector(vec3f v) {
    const float len = sqrt_(dot3(v, v));
    return mk(div_(v.x, len), div_(v.y, len), div_(v.z, len));
}

// ---- cuRAND XORWOW, subsequence 0 / offset 0 (curand_kernel.h:772-797,863-874; curand_uniform.h:69-72) --------
struct xorwow {
    uint32_t d, v0, v1, v2, v3, v4;
};
RT_HD void xorwow_seed(xorwow &s, unsigned long long seed) {
    const uint32_t s0 = (uint32_t)seed ^ 0xaad26b49u;
    const uint32_t s1 = (uint32_t)(seed >> 32) ^ 0xf7dcefddu;
    const uint32_t t0 = 1099087573u * s0;
    const uint32_t t1 = 2591861531u * s1;
    s.d = 6615241u + t1 + t0;
    s.v0 = 123456789u + t0;
    s.v1 = 362436069u ^ t0;
    s.v2 = 521288629u + t1;
    s.v3 = 88675123u ^ t1;
    s.v4 = 5783321u + t0;
}
RT_HD uint32_t xorwow_next(xorwow &s) {
    const uint32_t t = s.v0 ^ (s.v0 >> 2);
    s.v0 = s.v1; s.v1 = s.v2; s.v2 = s.v3; s.v3 = s.v4;
    s.v4 = (s.v4 ^ (s.v4 << 4)) ^ (t ^ (t << 1));
    s.d += 362437u;
    return s.v4 + s.d;
}
// (0, 1]: x * 2^-32 + 2^-33 (one FFMA on the device; the product is exact so fused == unfused)
RT_HD float xorwow_uniform(xorwow &s) {
    return fma_((float)xorwow_next(s), 2.3283064e-10f, 1.16415321826934814453125e-10f);
}

#if defined(__CUDACC__)
// A stream state in device memory: 6 words {d, v0..v4}, moved as three uint2, so the buffer must be 8-byte aligned (upstream
// seeds, progressive states, the per-ray queries' states).  The render kernels' start states are read by pixel_stream (__ldg).
__device__ __forceinline__ xorwow xorwow_load(const uint32_t *st) {
    const uint2 *s = reinterpret_cast<const uint2 *>(st);
    const uint2 a = s[0], b = s[1], c = s[2];
    xorwow rng;
    rng.d = a.x; rng.v0 = a.y; rng.v1 = b.x; rng.v2 = b.y; rng.v3 = c.x; rng.v4 = c.y;
    return rng;
}
__device__ __forceinline__ void xorwow_store(uint32_t *st, const xorwow &rng) {
    uint2 *o = reinterpret_cast<uint2 *>(st);
    o[0] = make_uint2(rng.d, rng.v0); o[1] = make_uint2(rng.v1, rng.v2); o[2] = make_uint2(rng.v3, rng.v4);
}
#endif

}  // namespace rt
