// Per-point arithmetic of the projection (reference src/encoding/range_image.py:146-198),
// written once for the device kernels and for the host-side test hook
// (nsc_test_host_classify) that lets the CPU-only test suite compare the pixel assignment
// with the oracle. No product path evaluates it on the host.
//
// What the reference computes per point, and what is computed here instead:
//   range   = sqrt((x*x + y*y) + z*z) in float32, kept iff 1 <= range <= 80  (:159-162,:174)
//             -> s = (x*x + y*y) + z*z formed with the same three roundings; kept iff
//                s_lo <= s <= s_hi where the two float32 thresholds are the exact preimages of
//                the range test under the correctly rounded sqrt (host_tables.cu). NaN / Inf
//                coordinates make s NaN / Inf and fail the test, which is the finite filter
//                (:151-155). The min over s is the min over range (sqrt is monotone); the
//                sqrt is taken once per pixel after the scatter.
//   column  = floor(((atan2(y,x) + pi) mod 2pi) / 2pi * 360)                       (:166-167,:194)
//             -> octant-reduced odd polynomial of atan in column units, error 3e-7 rad; the
//                north star excuses points within 1e-5 rad of a column edge. The reduction is
//                scale-invariant for every x, y with |x|, |y| < 2^64 -- signed zeros and
//                subnormals included, so points on or next to the vertical axis get the
//                reference's column -- which covers every point whose s is finite, i.e. every
//                point that can be kept. Larger or non-finite x, y still land in [0, 360].
//   row     = floor((atan2(z, sqrt(x*x+y*y)) - el_min) / (el_max - el_min) * E), clipped (:170,:186)
//             -> u = z / rho clamped to the field of view, odd polynomial of atan scaled to
//                row units (kRowPoly), or a binary search of z|z| against tan^2 thresholds
//                times rho^2 (kRowSearch, any field of view). Same 1e-5 rad excuse.
#pragma once
#include "nsc_internal.h"

#include <cmath>
#include <cstring>

#if defined(__CUDACC__)
#define NSC_HD __host__ __device__ __forceinline__
#else
#define NSC_HD inline
#endif

namespace nsc {

// atan(t) * 360 / (2 pi) = t * P(t^2) on [0, 1]: near-minimax fit (host_tables.cu fit_atan(1, 7)),
// max error 3.1e-7 rad in float32 Horner/FMA arithmetic, re-verified at library init. Literal
// constants so that every FFMA of the chain takes its coefficient as an immediate.
#define NSC_COL_C0 5.729555511e+01f
#define NSC_COL_C1 -1.908944511e+01f
#define NSC_COL_C2 1.134904289e+01f
#define NSC_COL_C3 -7.582146645e+00f
#define NSC_COL_C4 4.562099934e+00f
#define NSC_COL_C5 -1.925379395e+00f
#define NSC_COL_C6 3.902867138e-01f

// The device keeps floor() results as the raw bits of (v + 2^23) rounded down: the integer sits
// in the low mantissa bits above this bias, and the bias is folded into the address constant.
constexpr uint32_t kFloorBias = 0x4B000000u;

// float32 multiply / add with exactly one rounding each (no FMA contraction).
NSC_HD float mul_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    volatile float r = a * b;
    return r;
#endif
}
NSC_HD float add_rn(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    volatile float r = a + b;
    return r;
#endif
}
// MUFU.RCP / MUFU.RSQ on the device: one special-function op each, relative error <= 2^-22.
NSC_HD float rcp_fast(float a) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r;
#else
    return 1.0f / a;
#endif
}
NSC_HD float rsqrt_fast(float a) {
#if defined(__CUDA_ARCH__)
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r;
#else
    return 1.0f / sqrtf(a);
#endif
}
NSC_HD uint32_t f2u(float a) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(a);
#else
    uint32_t u;
    memcpy(&u, &a, 4);
    return u;
#endif
}

// floor(v + add) for v + add in [0, 2^22), plus kFloorBias (see above). On the device one FADD
// with round-down of the exact sum v + (add + 2^23); add must be an integer.
NSC_HD uint32_t floor_biased(float v, float add) {
#if defined(__CUDA_ARCH__)
    return __float_as_uint(__fadd_rd(v, add + 8388608.0f));
#else
    return (uint32_t)floor((double)v + (double)add) + kFloorBias;
#endif
}

// Octant reduction t = min(|x|,|y|) / max(|x|,|y|) with x and y first scaled by 2^32, which is
// exact: a nonzero magnitude below 2^64 (every x, y of a point whose s is finite) becomes a normal
// number in [2^-117, 2^96), where rcp.approx.ftz flushes neither its input nor its result, so t is
// the same for (x, y) and (2^k x, 2^k y), subnormals included. The floor only turns x = y = 0 into
// t = 0 (instead of 0 * Inf); it is below every scaled nonzero magnitude.
constexpr float kOctScale = 0x1p32f;
constexpr float kOctFloor = 0x1p-126f;

// |x| * 2^32 and |y| * 2^32; on the device one packed multiply (x and y of a loaded point sit in
// an aligned register pair).
NSC_HD void scaled_abs(float x, float y, float& ax, float& ay) {
#if defined(__CUDA_ARCH__)
    uint64_t v, k;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(x), "f"(y));
    asm("mov.b64 %0, {%1, %1};" : "=l"(k) : "f"(kOctScale));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(v) : "l"(v), "l"(k));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(ax), "=f"(ay) : "l"(v));
    ax = fabsf(ax);
    ay = fabsf(ay);
#else
    ax = fabsf(x * kOctScale);
    ay = fabsf(y * kOctScale);
#endif
}

// Column + kFloorBias, column in [0, 360]; 360 only for azimuth == 2*pi exactly, which the
// reference wraps to 0 (the kernels keep a 361st column and fold it).
NSC_HD uint32_t column_biased(float x, float y) {
    float ax, ay;
    scaled_abs(x, y, ax, ay);
    const float mx = fmaxf(fmaxf(ax, ay), kOctFloor);
    const float mn = fminf(ax, ay);
    const float t = mn * rcp_fast(mx);
    const float t2 = t * t;
    float p = NSC_COL_C6;
    p = fmaf(p, t2, NSC_COL_C5);
    p = fmaf(p, t2, NSC_COL_C4);
    p = fmaf(p, t2, NSC_COL_C3);
    p = fmaf(p, t2, NSC_COL_C2);
    p = fmaf(p, t2, NSC_COL_C1);
    p = fmaf(p, t2, NSC_COL_C0);
    float r = p * t;                                  // [0, 45] column units
    if (ay > ax) r = 90.0f - r;                       // |y| > |x|: reflect about the bisector
    if ((int32_t)f2u(x) < 0) r = 180.0f - r;          // sign BIT of x: atan2(+-0, -0) = +-pi
    r = copysignf(r, y);                              // sign bit of y
    r = fminf(r, 180.0f);                             // NaN (x and y both non-finite) -> in range
    return floor_biased(r, 180.0f);
}

// Row + kFloorBias. ROWS: the row capacity of the caller (a power of two >= E), which sets the
// depth of the kRowSearch binary search.
template <int ROWS = kShortRows, typename P>
NSC_HD uint32_t row_biased(float z, float rho2, const P& dp, int row_mode) {
    if (row_mode == kRowPoly) {
        float u = z * rsqrt_fast(rho2);               // rho2 == 0 -> +-inf, clamped below
        u = fminf(fmaxf(u, dp.u_lo), dp.u_hi);        // also maps NaN into the field of view
        const float u2 = u * u;
        float p = dp.row_p[kRowTerms - 1];
#pragma unroll
        for (int i = kRowTerms - 2; i >= 0; --i) p = fmaf(p, u2, dp.row_p[i]);
        return floor_biased(fmaf(p, u, dp.row_off), 0.0f);   // in (0, E) by construction of u_lo/u_hi
    }
    const float q = z * fabsf(z);
    int row = 0;
#pragma unroll
    for (int step = ROWS / 2; step > 0; step >>= 1) {
        const int k = row + step;
        if (k < dp.E && q >= dp.row_c[k] * rho2) row = k;
    }
    return (uint32_t)row + kFloorBias;
}

// One point -> biased row and column (always inside the kPitch-wide image, whatever the input)
// and the scatter key: the bits of s, or 0xffffffff (never a minimum) when s < s_lo. Keys above
// the bits of s_hi (too far, +Inf, NaN) are NOT filtered here: they can only survive in a pixel
// no in-range point hit, and the per-pixel conversion after the scatter maps them to "empty"
// (key_is_empty). That moves the upper half of the range filter from 120 k points to 5 760 pixels.
template <int ROWS = kShortRows, typename P>
NSC_HD uint32_t classify(float x, float y, float z, const P& dp, int row_mode, uint32_t& row_b,
                         uint32_t& col_b) {
    const float xx = mul_rn(x, x), yy = mul_rn(y, y), zz = mul_rn(z, z);
    const float rho2 = add_rn(xx, yy);
    const float s = add_rn(rho2, zz);
    col_b = column_biased(x, y);
    row_b = row_biased<ROWS>(z, rho2, dp, row_mode);
    return (s >= dp.s_lo) ? f2u(s) : 0xffffffffu;         // NaN compares false
}

#if defined(__CUDACC__)
// ---- two points at a time on the packed FP32 pipe (sm_100a FFMA2 / FMUL2) -----------------
// The polynomial parts of column_biased() / row_biased() for a PAIR of points evaluated with
// fma.rn.f32x2 / mul.rn.f32x2: every lane of a packed instruction rounds exactly like the scalar
// instruction, so classify2() returns bit for bit what two classify() calls return, in roughly
// 16 fewer issue slots per pair. The range sum keeps the scalar __fmul_rn/__fadd_rn (three
// separate roundings are part of the reference's result and must not be contracted).
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

template <int ROWS = kShortRows, typename P>
__device__ __forceinline__ void classify2(float xa, float ya, float za, float xb, float yb, float zb,
                                          const P& dp, int row_mode, uint32_t& key_a, uint32_t& row_a,
                                          uint32_t& col_a, uint32_t& key_b, uint32_t& row_b,
                                          uint32_t& col_b) {
    // range (scalar, exactly the reference's roundings)
    const float rho2a = __fadd_rn(__fmul_rn(xa, xa), __fmul_rn(ya, ya));
    const float rho2b = __fadd_rn(__fmul_rn(xb, xb), __fmul_rn(yb, yb));
    const float sa = __fadd_rn(rho2a, __fmul_rn(za, za));
    const float sb = __fadd_rn(rho2b, __fmul_rn(zb, zb));
    key_a = (sa >= dp.s_lo) ? __float_as_uint(sa) : 0xffffffffu;
    key_b = (sb >= dp.s_lo) ? __float_as_uint(sb) : 0xffffffffu;
    // column: octant reduction (scaled as in column_biased) scalar, polynomial packed
    float axa, aya, axb, ayb;
    scaled_abs(xa, ya, axa, aya);
    scaled_abs(xb, yb, axb, ayb);
    const float ra = rcp_fast(fmaxf(fmaxf(axa, aya), kOctFloor)), rb = rcp_fast(fmaxf(fmaxf(axb, ayb), kOctFloor));
    const uint64_t t = mul2(pack2(fminf(axa, aya), fminf(axb, ayb)), pack2(ra, rb));
    const uint64_t t2 = mul2(t, t);
    uint64_t p = pack2(NSC_COL_C6, NSC_COL_C6);
    p = fma2(p, t2, pack2(NSC_COL_C5, NSC_COL_C5));
    p = fma2(p, t2, pack2(NSC_COL_C4, NSC_COL_C4));
    p = fma2(p, t2, pack2(NSC_COL_C3, NSC_COL_C3));
    p = fma2(p, t2, pack2(NSC_COL_C2, NSC_COL_C2));
    p = fma2(p, t2, pack2(NSC_COL_C1, NSC_COL_C1));
    p = fma2(p, t2, pack2(NSC_COL_C0, NSC_COL_C0));
    float ca, cb;
    unpack2(mul2(p, t), ca, cb);
    if (aya > axa) ca = 90.0f - ca;
    if (ayb > axb) cb = 90.0f - cb;
    if ((int32_t)__float_as_uint(xa) < 0) ca = 180.0f - ca;
    if ((int32_t)__float_as_uint(xb) < 0) cb = 180.0f - cb;
    ca = fminf(copysignf(ca, ya), 180.0f);
    cb = fminf(copysignf(cb, yb), 180.0f);
    col_a = floor_biased(ca, 180.0f);
    col_b = floor_biased(cb, 180.0f);
    // row
    if (row_mode == kRowPoly) {
        float ua, ub;
        unpack2(mul2(pack2(za, zb), pack2(rsqrt_fast(rho2a), rsqrt_fast(rho2b))), ua, ub);
        ua = fminf(fmaxf(ua, dp.u_lo), dp.u_hi);
        ub = fminf(fmaxf(ub, dp.u_lo), dp.u_hi);
        const uint64_t u = pack2(ua, ub);
        const uint64_t u2 = mul2(u, u);
        uint64_t q = pack2(dp.row_p[kRowTerms - 1], dp.row_p[kRowTerms - 1]);
#pragma unroll
        for (int i = kRowTerms - 2; i >= 0; --i) q = fma2(q, u2, pack2(dp.row_p[i], dp.row_p[i]));
        float va, vb;
        unpack2(fma2(q, u, pack2(dp.row_off, dp.row_off)), va, vb);
        row_a = floor_biased(va, 0.0f);
        row_b = floor_biased(vb, 0.0f);
    } else {
        row_a = row_biased<ROWS>(za, rho2a, dp, row_mode);
        row_b = row_biased<ROWS>(zb, rho2b, dp, row_mode);
    }
}
#endif

// A pixel key that no kept point produced: the initial +Inf, or a point beyond max range / NaN.
template <typename P>
NSC_HD bool key_is_empty(uint32_t key, const P& dp) { return key > f2u(dp.s_hi); }

}  // namespace nsc
