// ccu_math.cuh - fp32 vector helpers and the deterministic transcendental set ("detmath").
//
// Arithmetic contract (DESIGN.md): every fp32 operation the reference writes out is one IEEE-754
// round-to-nearest operation in the order written; the OpenCL vector builtins expand as NVIDIA's runtime does.  The translation unit is compiled with -fmad=false (no contraction), default
// -prec-div=true -prec-sqrt=true -ftz=false.  sin/cos/atan2/asin/acos are fixed polynomial kernels built
// from +,-,*,/,sqrt,floor only, so the full path - not just the integer first-hit buffers - reproduces
// bit-for-bit on any IEEE machine.  (The reference calls the OpenCL builtins cos/sin/atan2/asin/acos,
// sky.h:26-37,51-53,80-82,99-103, kernel.h:57-59, camera.h:26-27, whose results are implementation
// defined to a few ulp; detmath stays within 2 ulp of them on the ranges used - tests/test_math.py.)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace ccu {

#define CCU_EPS 0.000005f    // constants.h:4
#define CCU_OFFSET 0.0001f   // constants.h:5
#define CCU_PI_F 3.14159274101257f
#define CCU_PI_2_F 1.57079637050629f
#define CCU_INV_PI_F 0.318309886183791f

__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
// dot / cross / normalize stand for the OpenCL builtins of the same name and are expanded exactly as the
// NVIDIA OpenCL runtime expands them (explicit fused multiply-adds; PTX evidence: profiles/clref_vec_strict.ptx).
__device__ __forceinline__ float dot3(float3 a, float3 b) { return __fmaf_rn(a.z, b.z, __fmaf_rn(a.x, b.x, a.y * b.y)); }
__device__ __forceinline__ float3 cross3(float3 a, float3 b) {
    return f3(__fmaf_rn(a.y, b.z, -(a.z * b.y)), __fmaf_rn(a.z, b.x, -(a.x * b.z)), __fmaf_rn(a.x, b.y, -(a.y * b.x)));
}
// One division site per role (scale, divide, second divide) instead of one per return path: the operations a given input goes
// through are the same ones in the same order (v / inf for an infinite component; v / (m * r) normally; (v / r) / m when m * r
// overflows), the quotients of the paths not taken are computed on the side and dropped.
__device__ __forceinline__ float3 normalize3(float3 v) {
    const float inf = __int_as_float(0x7f800000), qnan = __int_as_float(0x7fc00000);
    float ax = fabsf(v.x), ay = fabsf(v.y), az = fabsf(v.z);
    if (ax != ax || ay != ay || az != az) return f3(qnan, qnan, qnan);
    float m = (ax < ay) ? ay : ax;
    m = (m < az) ? az : m;
    if (m == 0.0f) return f3(0, 0, 0);
    float a = ax / m, b = ay / m, c = az / m;
    float r = sqrtf(__fmaf_rn(c, c, __fmaf_rn(a, a, b * b)));
    float len = m * r;
    const bool by_inf = m == inf;                       // v / inf
    const bool two_step = !by_inf && !(fabsf(len) != inf);   // (v / r) / m
    const float d1 = by_inf ? inf : (two_step ? r : len);
    float3 q = f3(v.x / d1, v.y / d1, v.z / d1);
    if (two_step) q = f3(q.x / m, q.y / m, q.z / m);
    return q;
}
// cvt.rzi.s32.f32: toward zero, saturating, NaN -> 0
__device__ __forceinline__ int f2i(float f) { return __float2int_rz(f); }
__device__ __forceinline__ float i2f(int bits) { return __int_as_float(bits); }
__device__ __forceinline__ bool is_nan(float f) { return f != f; }
__device__ __forceinline__ float nanf_() { return __int_as_float(0x7fc00000); }
__device__ __forceinline__ float inff_() { return __int_as_float(0x7f800000); }

// (sin x, cos x) in one evaluation
__device__ __forceinline__ float2 dm_sincos2(float x) {
    float s, c;
    float kf = floorf(x * 0.636619772f + 0.5f);
    float r = x - kf * 1.5703125f;
    r = r - kf * 4.837512969970703125e-4f;
    r = r - kf * 7.54978995489188216e-8f;
    int k = f2i(kf) & 3;
    float z = r * r;
    float sp = ((-1.9515295891e-4f * z + 8.3321608736e-3f) * z - 1.6666654611e-1f) * z * r + r;
    float cp = ((2.443315711809948e-5f * z - 1.388731625493765e-3f) * z + 4.166664568298827e-2f) * z * z - 0.5f * z + 1.0f;
    float ss = (k & 1) ? cp : sp;
    float cc = (k & 1) ? sp : cp;
    s = (k & 2) ? -ss : ss;
    c = ((k + 1) & 2) ? -cc : cc;
    return make_float2(s, c);
}
__device__ __forceinline__ void dm_sincos(float x, float &s, float &c) { const float2 r = dm_sincos2(x); s = r.x; c = r.y; }
__device__ __forceinline__ float dm_cos(float x) { float s, c; dm_sincos(x, s, c); return c; }
__device__ __forceinline__ float dm_sin(float x) { float s, c; dm_sincos(x, s, c); return s; }

// One division, one polynomial: -(1 / t) == (-1) / t bit for bit (round-to-nearest is sign-symmetric), so both range
// reductions are num / den with selected operands.
__device__ __forceinline__ float dm_atan(float t) {
    float sign = 1.0f, y0 = 0.0f;
    if (t < 0.0f) { t = -t; sign = -1.0f; }
    const bool big = t > 2.414213562373095f, mid = !big && t > 0.4142135623730950f;
    if (big) y0 = 1.5707963267948966f;
    if (mid) y0 = 0.7853981633974483f;
    if (big || mid) t = (big ? -1.0f : t - 1.0f) / (big ? t : t + 1.0f);
    float z = t * t;
    float p = (((8.05374449538e-2f * z - 1.38776856032e-1f) * z + 1.99777106478e-1f) * z - 3.33329491539e-1f) * z * t + t;
    return sign * (y0 + p);
}
// one dm_atan site: the quadrant offset is added afterwards (x > 0: none; x < 0: +pi for y >= 0, -pi for y < 0)
__device__ __forceinline__ float dm_atan2(float y, float x) {
    if (x != x || y != y) return nanf_();
    if (x == 0.0f) return y > 0.0f ? 1.5707963267948966f : (y < 0.0f ? -1.5707963267948966f : 0.0f);
    const float a = dm_atan(y / x);
    if (x > 0.0f) return a;
    return (y >= 0.0f) ? a + 3.14159265358979f : a - 3.14159265358979f;
}
__device__ __forceinline__ float dm_asin(float x) {
    float a = fabsf(x);
    if (a > 1.0f) return nanf_();
    bool big = a > 0.5f;
    float z, t;
    if (big) { z = 0.5f * (1.0f - a); t = sqrtf(z); } else { t = a; z = t * t; }
    float p = ((((4.2163199048e-2f * z + 2.4181311049e-2f) * z + 4.5470025998e-2f) * z + 7.4953002686e-2f) * z + 1.6666752422e-1f) * z * t + t;
    if (big) p = 1.5707963267948966f - (p + p);
    return x < 0.0f ? -p : p;
}
// one dm_asin site: 1 + x == 1 - |x| for x < -0.5 and 1 - x == 1 - |x| for x > 0.5 (a + b == a - (-b) exactly)
__device__ __forceinline__ float dm_acos(float x) {
    if (fabsf(x) > 1.0f) return nanf_();
    const bool lo = x < -0.5f, hi = x > 0.5f;
    const float arg = (lo || hi) ? sqrtf(0.5f * (1.0f - fabsf(x))) : x;
    const float as = dm_asin(arg);
    if (lo) return 3.14159265358979f - 2.0f * as;
    if (hi) return 2.0f * as;
    return 1.5707963267948966f - as;
}

// e^x as a fixed kernel (the fog's transmittance, DESIGN §14), built like dm_powf (ccu_tonemap.cuh): an fp64 series from
// + - * / only, rounded once to fp32, so that the CPU restatement evaluates the same bits.  exp(-inf) = 0, exp(NaN) = NaN.
__device__ __forceinline__ float dm_expf(float x) {
    if (x != x) return nanf_();
    if (x > 89.0f) return inff_();
    if (x < -104.0f) return 0.0f;                                   // e^-104 < 2^-150: rounds to 0
    const double p = (double)x * 1.4426950408889634;                // log2 e
    const double k = floor(p + 0.5);
    const double f = (p - k) * 0.6931471805599453;                  // ln 2, |f| <= 0.3466
    double r = 1.0 / 479001600.0;                                   // exp(f), Taylor to f^12
    r = r * f + 1.0 / 39916800.0;
    r = r * f + 1.0 / 3628800.0;
    r = r * f + 1.0 / 362880.0;
    r = r * f + 1.0 / 40320.0;
    r = r * f + 1.0 / 5040.0;
    r = r * f + 1.0 / 720.0;
    r = r * f + 1.0 / 120.0;
    r = r * f + 1.0 / 24.0;
    r = r * f + 1.0 / 6.0;
    r = r * f + 0.5;
    r = r * f + 1.0;
    r = r * f + 1.0;
    const double scale = __longlong_as_double((long long)((int)k + 1023) << 52);   // 2^k, -151 <= k <= 129
    return (float)(r * scale);
}

// 256-bit read-only global load (LDG.E.256 on sm_100a): one instruction and one L1 tag lookup per lane for a 32-byte record half
struct __align__(32) Int8 { int v[8]; };
__device__ __forceinline__ Int8 ldg256(const void *p) {
    Int8 r;
    asm volatile("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r.v[0]), "=r"(r.v[1]), "=r"(r.v[2]), "=r"(r.v[3]), "=r"(r.v[4]), "=r"(r.v[5]), "=r"(r.v[6]), "=r"(r.v[7])
                 : "l"(p));
    return r;
}

// PCG hash RNG: randomness.h:6-17
__device__ __forceinline__ uint32_t rng_next(uint32_t &state) {
    uint32_t s = state * 47796405u + 2891336453u;
    s = ((s >> ((s >> 28u) + 4u)) ^ s) * 277803737u;
    s = (s >> 22u) ^ s;
    state = s;
    return s;
}
__device__ __forceinline__ float rng_float(uint32_t &state) { return (float)(rng_next(state) >> 8) / 16777216.0f; }

}  // namespace ccu
