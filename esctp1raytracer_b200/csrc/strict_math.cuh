// strict_math.cuh — the reference's arithmetic, bit for bit, on the device.
//
// The reference serial path is built for baseline x86-64: every float
// operation rounds once (SSE scalar, no FMA contraction).  Its image is
// numerically chaotic (shadow rays start ON the surface, src/main.cpp:757-758),
// so every decision and every value that reaches the framebuffer is evaluated
// here with correctly-rounded intrinsics, which nvcc never contracts:
//   a*b -> __fmul_rn   a+b -> __fadd_rn   a-b -> __fsub_rn
//   a/b -> __fdiv_rn   sqrtf -> __fsqrt_rn
//   double det / inv_det of ray_triangle.h:21-26 -> real FP64 (__ddiv_rn, __dmul_rn)
//   libm powf of the shading (main.cpp:783) -> powf_glibc below (glibc's own algorithm, op for op)
// The O(N) sweeps run a cheap conservative filter instead (sweep.cuh) and
// only the surviving (ray, triangle) pairs come through these functions.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <cuda_runtime.h>

namespace strict {

#define TRC_EPS 1.1920928955078125e-07f /* std::numeric_limits<float>::epsilon() */

struct f3 {
    float x, y, z;
};

__device__ __forceinline__ f3 mk(float x, float y, float z) {
    f3 r;
    r.x = x, r.y = y, r.z = z;
    return r;
}
__device__ __forceinline__ f3 ld(const float *p) { return mk(p[0], p[1], p[2]); }

// vec.h:95-101 — sum starts at 0 and accumulates left to right
__device__ __forceinline__ float dot(f3 a, f3 b) {
    float s = __fadd_rn(0.f, __fmul_rn(a.x, b.x));
    s = __fadd_rn(s, __fmul_rn(a.y, b.y));
    s = __fadd_rn(s, __fmul_rn(a.z, b.z));
    return s;
}
// vec.h:103-109
__device__ __forceinline__ f3 cross(f3 a, f3 b) {
    return mk(__fsub_rn(__fmul_rn(a.y, b.z), __fmul_rn(a.z, b.y)), __fsub_rn(__fmul_rn(a.z, b.x), __fmul_rn(a.x, b.z)),
              __fsub_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
}
__device__ __forceinline__ f3 add(f3 a, f3 b) { return mk(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y), __fadd_rn(a.z, b.z)); }
__device__ __forceinline__ f3 sub(f3 a, f3 b) { return mk(__fsub_rn(a.x, b.x), __fsub_rn(a.y, b.y), __fsub_rn(a.z, b.z)); }
__device__ __forceinline__ f3 mul(f3 a, float s) { return mk(__fmul_rn(a.x, s), __fmul_rn(a.y, s), __fmul_rn(a.z, s)); }
__device__ __forceinline__ f3 div(f3 a, float s) { return mk(__fdiv_rn(a.x, s), __fdiv_rn(a.y, s), __fdiv_rn(a.z, s)); }
// vec.h:135-139
__device__ __forceinline__ float length(f3 a) { return __fsqrt_rn(dot(a, a)); }
__device__ __forceinline__ f3 normalize(f3 a) { return div(a, __fsqrt_rn(dot(a, a))); }

// tracer::intersect_triangle, src/scene/ray_triangle.h:7-57.
// On accept: t <- t2, v <- v2 (the caller's u aliases v, src/main.cpp:307/310,
// so only v survives) and returns true.
__device__ __forceinline__ bool intersect_triangle(f3 orig, f3 dir, f3 vert0, f3 vert1, f3 vert2, float &t, float &v) {
    const f3 edge1 = sub(vert1, vert0);
    const f3 edge2 = sub(vert2, vert0);
    const f3 pvec = cross(dir, edge2);
    const double det = (double)dot(edge1, pvec);
    if (det > -(double)TRC_EPS && det < (double)TRC_EPS) return false;
    const double inv_det = __ddiv_rn(1.0, det);
    const f3 tvec = sub(orig, vert0);
    const float u2 = __double2float_rn(__dmul_rn((double)dot(tvec, pvec), inv_det));
    if (u2 < TRC_EPS || u2 > 1.0f) return false;
    const f3 qvec = cross(tvec, edge1);
    const float v2 = __double2float_rn(__dmul_rn((double)dot(dir, qvec), inv_det));
    if (v2 < TRC_EPS || __fadd_rn(u2, v2) > 1.0f) return false;
    const float t2 = __double2float_rn(__dmul_rn((double)dot(edge2, qvec), inv_det));
    if (t2 < TRC_EPS) return false;
    if (t2 >= t) return false;
    t = t2;
    v = v2;
    return true;
}

// Extension with no reference code (src/intersect.h is empty): analytic
// ray-sphere for unit-length dir; same epsilon rules as the triangle test.
// Mirrors oracle/restated.c:sphere_test op for op.
__device__ __forceinline__ bool intersect_sphere(f3 orig, f3 dir, float4 cr, float &t) {
    const f3 oc = sub(orig, mk(cr.x, cr.y, cr.z));
    const float b = dot(oc, dir);
    const float c = __fsub_rn(dot(oc, oc), __fmul_rn(cr.w, cr.w));
    const float disc = __fsub_rn(__fmul_rn(b, b), c);
    if (!(disc >= 0.f)) return false;
    const float sq = __fsqrt_rn(disc);
    float t2 = __fsub_rn(-b, sq);
    if (t2 < TRC_EPS) t2 = __fadd_rn(-b, sq);
    if (t2 < TRC_EPS) return false;
    if (t2 >= t) return false;
    t = t2;
    return true;
}

// ---------------------------------------------------------------------------------------------------------------------
// powf exactly as the reference's libm computes it (the shading's powf(dot(N,H), Ns), main.cpp:783).
//
// glibc >= 2.28 ships Arm optimized-routines' powf (math/powf.c, Copyright (c) 2017-2018 Arm Limited, MIT OR
// Apache-2.0 WITH LLVM-exception): log2(x) from a 16-entry (1/c, log2 c) table and a degree-5 polynomial, y*log2(x)
// in double, 2^that from a 32-entry table and a degree-3 polynomial.  It is NOT correctly rounded (not even for
// y = 2), so neither the device's pow nor (float)pow((double)x, (double)y) reproduces it.  On x86-64 glibc builds it
// twice and picks one at load time (ifunc): plain SSE2, or -mfma -mavx2, where GCC contracts every a*b+c into one
// FMA.  The two disagree on rare inputs.  This port is the FMA variant, the one x86-64 hosts with FMA + AVX2 run,
// read off the machine code of glibc 2.39's libm: its contractions are the pw_fma calls below, its constants are
// the tables' bits.  Every double operation is an explicit correctly-rounded intrinsic, so nvcc cannot contract or
// reorder anything and the host build (tests/strict_host_shim.cpp) is the same sequence of operations.
// Special cases (x subnormal / zero / negative / inf / NaN, y zero / inf / NaN, overflow, underflow) follow glibc's
// branches; results with errno side effects return the value glibc returns in round-to-nearest.
#ifdef __CUDACC__
#define STRICT_TABLE __constant__
#else
#define STRICT_TABLE
#endif
// {1/c, log2(c)}, c near the middle of subinterval i of the reduced argument z in [OFF, 2 OFF), OFF = 0x3f330000 as
// float bits (about 0.7); i = the top 4 mantissa bits of z - OFF
STRICT_TABLE static const double POWF_LOG2_TAB[16][2] = {
    {0x1.661ec79f8f3bep+0, -0x1.efec65b963019p-2}, {0x1.571ed4aaf883dp+0, -0x1.b0b6832d4fca4p-2},
    {0x1.49539f0f010bp+0, -0x1.7418b0a1fb77bp-2},  {0x1.3c995b0b80385p+0, -0x1.39de91a6dcf7bp-2},
    {0x1.30d190c8864a5p+0, -0x1.01d9bf3f2b631p-2}, {0x1.25e227b0b8eap+0, -0x1.97c1d1b3b7afp-3},
    {0x1.1bb4a4a1a343fp+0, -0x1.2f9e393af3c9fp-3}, {0x1.12358f08ae5bap+0, -0x1.960cbbf788d5cp-4},
    {0x1.0953f419900a7p+0, -0x1.a6f9db6475fcep-5}, {0x1p+0, 0x0p+0},
    {0x1.e608cfd9a47acp-1, 0x1.338ca9f24f53dp-4},  {0x1.ca4b31f026aap-1, 0x1.476a9543891bap-3},
    {0x1.b2036576afce6p-1, 0x1.e840b4ac4e4d2p-3},  {0x1.9c2d163a1aa2dp-1, 0x1.40645f0c6651cp-2},
    {0x1.886e6037841edp-1, 0x1.88e9c2c1b9ff8p-2},  {0x1.767dcf5534862p-1, 0x1.ce0a44eb17bccp-2},
};
// bits of 2^(i/32) minus i << 47 (the exponent is added back from the integer part of the argument)
STRICT_TABLE static const uint64_t POWF_EXP2_TAB[32] = {
    0x3ff0000000000000, 0x3fefd9b0d3158574, 0x3fefb5586cf9890f, 0x3fef9301d0125b51, 0x3fef72b83c7d517b, 0x3fef54873168b9aa,
    0x3fef387a6e756238, 0x3fef1e9df51fdee1, 0x3fef06fe0a31b715, 0x3feef1a7373aa9cb, 0x3feedea64c123422, 0x3feece086061892d,
    0x3feebfdad5362a27, 0x3feeb42b569d4f82, 0x3feeab07dd485429, 0x3feea47eb03a5585, 0x3feea09e667f3bcd, 0x3fee9f75e8ec5f74,
    0x3feea11473eb0187, 0x3feea589994cce13, 0x3feeace5422aa0db, 0x3feeb737b0cdc5e5, 0x3feec49182a3f090, 0x3feed503b23e255d,
    0x3feee89f995ad3ad, 0x3feeff76f2fb5e47, 0x3fef199bdd85529c, 0x3fef3720dcef9069, 0x3fef5818dcfba487, 0x3fef7c97337b9b5f,
    0x3fefa4afa2a490da, 0x3fefd0765b6e4540,
};

// The double additions and fused multiply-adds of powf_glibc: correctly-rounded intrinsics on the device; in a host
// build of this header (compiled without FP contraction) the IEEE operations they are defined as.
__device__ __forceinline__ double pw_add(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
__device__ __forceinline__ double pw_sub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
__device__ __forceinline__ double pw_fma(double a, double b, double c) {
#ifdef __CUDA_ARCH__
    return __fma_rn(a, b, c);
#else
    return std::fma(a, b, c);
#endif
}

__device__ __forceinline__ uint32_t pw_asuint(float f) { uint32_t u; memcpy(&u, &f, sizeof u); return u; }
__device__ __forceinline__ float pw_asfloat(uint32_t u) { float f; memcpy(&f, &u, sizeof f); return f; }
__device__ __forceinline__ uint64_t pw_asuint64(double d) { uint64_t u; memcpy(&u, &d, sizeof u); return u; }
__device__ __forceinline__ double pw_asdouble(uint64_t u) { double d; memcpy(&d, &u, sizeof d); return d; }

// log2(x) for the bits of a positive normal x (or of a subnormal x scaled by 2^23 with its exponent lowered by 23)
__device__ __forceinline__ double powf_log2_inline(uint32_t ix) {
    const uint32_t tmp = ix - 0x3f330000u;
    const int i = (int)((tmp >> 19) % 16);
    const uint32_t top = tmp & 0xff800000u;
    const uint32_t iz = ix - top;
    const int k = (int32_t)top >> 23; // arithmetic shift
    const double invc = POWF_LOG2_TAB[i][0], logc = POWF_LOG2_TAB[i][1];
    const double z = (double)pw_asfloat(iz);
    // log2(x) = log1p(z/c-1)/ln2 + log2(c) + k
    const double r = pw_fma(z, invc, -1.0);
    const double y0 = pw_add(logc, (double)k);
    const double r2 = __dmul_rn(r, r);
    const double y = pw_fma(0x1.27616c9496e0bp-2, r, -0x1.71969a075c67ap-2);
    const double p = pw_fma(0x1.ec70a6ca7baddp-2, r, -0x1.7154748bef6c8p-1);
    const double r4 = __dmul_rn(r2, r2);
    double q = pw_fma(0x1.71547652ab82bp+0, r, y0);
    q = pw_fma(p, r2, q);
    return pw_fma(y, r4, q);
}

// 2^xd for -150 < xd <= 128; sign_bias = 1 << 16 flips the sign of the result
__device__ __forceinline__ float powf_exp2_inline(double xd, uint64_t sign_bias) {
    const double shift = 0x1.8p+52 / 32;
    double kd = pw_add(xd, shift); // xd = k/32 + r, r in [-1/64, 1/64]
    const uint64_t ki = pw_asuint64(kd);
    kd = pw_sub(kd, shift);
    const double r = pw_sub(xd, kd);
    // 2^xd = 2^(k/32) * 2^r ~= s * (C0*r^3 + C1*r^2 + C2*r + 1)
    uint64_t t = POWF_EXP2_TAB[ki % 32];
    t += (ki + sign_bias) << 47;
    const double s = pw_asdouble(t);
    const double z = pw_fma(0x1.c6af84b912394p-5, r, 0x1.ebfce50fac4f3p-3);
    const double r2 = __dmul_rn(r, r);
    double y = pw_fma(0x1.62e42ff0c52d6p-1, r, 1.0);
    y = pw_fma(z, r2, y);
    y = __dmul_rn(y, s);
    return __double2float_rn(y);
}

// 0: y is not an integer, 1: odd integer, 2: even integer (iy: bits of a non-zero finite y)
__device__ __forceinline__ int powf_checkint(uint32_t iy) {
    const int e = iy >> 23 & 0xff;
    if (e < 0x7f) return 0;
    if (e > 0x7f + 23) return 2;
    if (iy & ((1u << (0x7f + 23 - e)) - 1)) return 0;
    if (iy & (1u << (0x7f + 23 - e))) return 1;
    return 2;
}
__device__ __forceinline__ bool powf_zeroinfnan(uint32_t i) { return 2u * i - 1u >= 2u * 0x7f800000u - 1u; }
__device__ __forceinline__ bool powf_issignaling(uint32_t i) { return ((i ^ 0x00400000u) & 0x7fffffffu) > 0x7fc00000u; }

__device__ __forceinline__ float powf_glibc(float x, float y) {
    uint64_t sign_bias = 0;
    uint32_t ix = pw_asuint(x);
    const uint32_t iy = pw_asuint(y);
    if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u || powf_zeroinfnan(iy)) {
        // x < 0x1p-126 or inf or nan, or y is 0 or inf or nan
        if (powf_zeroinfnan(iy)) {
            if (2u * iy == 0) return powf_issignaling(ix) ? __fadd_rn(x, y) : 1.0f;
            if (ix == 0x3f800000u) return powf_issignaling(iy) ? __fadd_rn(x, y) : 1.0f;
            if (2u * ix > 2u * 0x7f800000u || 2u * iy > 2u * 0x7f800000u) return __fadd_rn(x, y);
            if (2u * ix == 2u * 0x3f800000u) return 1.0f;
            if ((2u * ix < 2u * 0x3f800000u) == !(iy & 0x80000000u)) return 0.0f; // |x|<1 && y==inf or |x|>1 && y==-inf
            return __fmul_rn(y, y);
        }
        if (powf_zeroinfnan(ix)) {
            float x2 = __fmul_rn(x, x);
            if ((ix & 0x80000000u) && powf_checkint(iy) == 1) x2 = -x2;
            return (iy & 0x80000000u) ? __fdiv_rn(1.0f, x2) : x2; // 1/(+-0) is glibc's divide-by-zero result too
        }
        // x and y are non-zero finite
        if (ix & 0x80000000u) {
            const int yint = powf_checkint(iy);
            if (yint == 0) return __fdiv_rn(__fsub_rn(x, x), __fsub_rn(x, x)); // invalid: NaN
            if (yint == 1) sign_bias = 1u << 16;
            ix &= 0x7fffffffu;
        }
        if (ix < 0x00800000u) { // subnormal x: scale to normal, then put the 23 back into the exponent field
            ix = pw_asuint(__fmul_rn(pw_asfloat(ix), 0x1p23f)) & 0x7fffffffu;
            ix -= 23u << 23;
        }
    }
    const double logx = powf_log2_inline(ix);
    const double ylogx = __dmul_rn((double)y, logx); // cannot overflow: y is a float
    if ((pw_asuint64(ylogx) >> 47 & 0xffff) >= pw_asuint64(126.0) >> 47) {
        // |y*log2(x)| >= 126
        if (ylogx > 0x1.fffffffd1d571p+6) return sign_bias ? -INFINITY : INFINITY; // overflow
        // (between 0x1.fffffffa3aae2p+6 and there glibc only checks for a directed rounding mode)
        if (ylogx <= -150.0) return sign_bias ? -0.0f : 0.0f;                 // underflow
        if (ylogx < -149.0) return sign_bias ? -0x1p-149f : 0x1p-149f;        // glibc's may-underflow value, 0x1.4p-75f^2
    }
    return powf_exp2_inline(ylogx, sign_bias);
}

}  // namespace strict
