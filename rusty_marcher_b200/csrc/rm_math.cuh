// rm_math.cuh -- scalar/vector helpers of the render kernels.
//
// Two numeric policies share one code base (template parameter R):
//   R = double : the reference's f64 arithmetic restated operation for operation
//                (engine/src/geometry.rs:18-182): left-to-right dot products, NO fused
//                multiply-add (the translation unit is compiled with -fmad=false), IEEE sqrt
//                and division.  This is the validation mode (RM_FP64).
//   R = float  : production mode.  Every multiply-add is an explicit fmaf() so the FP32
//                pipe issues one FFMA where the reference spends a mul and an add; nothing is
//                left to the compiler's contraction heuristics (-fmad=false).
#pragma once

#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define RM_HD __host__ __device__ __forceinline__
#define RM_D __device__ __forceinline__
#else
#define RM_HD inline
#define RM_D inline
#endif

namespace rm {

template <typename R> struct alignas(4 * sizeof(R)) R4 { R x, y, z, w; };
template <typename R> struct alignas(2 * sizeof(R)) R2 { R x, y; };
struct alignas(8) I2 { int x, y; };

template <typename R> struct Vec3 { R x, y, z; };

template <typename R> struct Num;

template <> struct Num<double> {
    static RM_HD double madd(double a, double b, double c) { return a * b + c; }     // unfused (-fmad=false)
    static RM_HD double msub(double a, double b, double c) { return a * b - c; }
    static RM_HD double nmadd(double a, double b, double c) { return c - a * b; }
    static RM_HD double sqrt_(double a) { return sqrt(a); }
    static RM_HD double abs_(double a) { return fabs(a); }
    static RM_HD double max_(double a, double b) { return fmax(a, b); }
    static RM_HD double pow_(double a, double b) { return pow(a, b); }
    static RM_HD double div_(double a, double b) { return a / b; }
    static RM_HD double rcp_(double a) { return 1. / a; }
};

// FP32 fast-math primitives of the production path (device: MUFU-based, host emulation: libm).
#if defined(__CUDA_ARCH__)
// a/b as a * rcp(b) without the denormal rescue sequence; callers guarantee |b| is a normal number
RM_HD float fast_div(float a, float b) {
    float r;
    asm("div.approx.ftz.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
// MUFU.RSQ (2 ulp) + one Newton step: 1/sqrt(a) to ~1 ulp in four instructions instead of IEEE sqrt + IEEE divide.
// rsqrt.approx.ftz is the bare MUFU (rsqrtf() wraps it in a rescue sequence for subnormal arguments; the arguments here
// are squared lengths of scene-scale vectors).
RM_HD float fast_rsqrt(float a) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));
    return r * fmaf(-0.5f * a * r, r, 1.5f);
}
#else
RM_HD float fast_div(float a, float b) { return a / b; }
RM_HD float fast_rsqrt(float a) { return 1.f / sqrtf(a); }
#endif

// x^e for x >= 0.  The specular exponents of the reference are small integers (30 in
// Reflectance::create_default, shapes.rs:55; 10..100 in scene.rs), for which square-and-multiply is both
// cheaper (about 15 FMULs) and more accurate (<= e * 2^-24 relative) than a generic powf; anything else
// takes the library routine.
RM_HD float pow_nonneg(float x, float e) {
    const int n = (int)e;
    if ((float)n == e && n >= 0 && n <= 1024) {
        float r = 1.f;
        // the two exponents the reference's scenes use most (30: Reflectance::create_default, shapes.rs:55; 100: scene.rs)
        // by their shortest addition chains: 6 and 8 multiplications
        if (n == 30) {
            const float x2 = x * x, x3 = x2 * x, x5 = x3 * x2, x10 = x5 * x5, x15 = x10 * x5;
            return x15 * x15;
        }
        if (n == 100) {
            const float x2 = x * x, x3 = x2 * x, x6 = x3 * x3, x12 = x6 * x6, x24 = x12 * x12, x25 = x24 * x, x50 = x25 * x25;
            return x50 * x50;
        }
        if (n < 128) {
            // straight-line square-and-multiply: six squarings, then the factors picked by the bits of n (no loop
            // counter, no branch; n is the same for every pixel of a material)
            const float x2 = x * x, x4 = x2 * x2, x8 = x4 * x4, x16 = x8 * x8, x32 = x16 * x16, x64 = x32 * x32;
            if (n & 1) r *= x;
            if (n & 2) r *= x2;
            if (n & 4) r *= x4;
            if (n & 8) r *= x8;
            if (n & 16) r *= x16;
            if (n & 32) r *= x32;
            if (n & 64) r *= x64;
            return r;
        }
        for (int k = n; k; k >>= 1) {
            if (k & 1) r *= x;
            x *= x;
        }
        return r;
    }
    return powf(x, e);
}

template <> struct Num<float> {
    static RM_HD float madd(float a, float b, float c) { return fmaf(a, b, c); }
    static RM_HD float msub(float a, float b, float c) { return fmaf(a, b, -c); }
    static RM_HD float nmadd(float a, float b, float c) { return fmaf(-a, b, c); }
    static RM_HD float sqrt_(float a) { return sqrtf(a); }
    static RM_HD float abs_(float a) { return fabsf(a); }
    static RM_HD float max_(float a, float b) { return fmaxf(a, b); }
    static RM_HD float pow_(float a, float b) { return pow_nonneg(a, b); }
    static RM_HD float div_(float a, float b) { return a / b; }
    static RM_HD float rcp_(float a) { return 1.f / a; }
};

// f64 at FP32 cost where 1e-14 is as good as 1e-16 (the glass paths of the production kernel, cast_glass<double> in
// rm_fast.cuh -- NOT the RM_FP64 validation kernels, which keep IEEE sqrt and division): an FP32 seed (MUFU) and one
// Newton step in f64 -- five f64 operations instead of the thirty-odd of the IEEE sequences.  Arguments are squared
// lengths, cosines and refractive indices: well inside the FP32 range.
struct Fast64 {
    static RM_HD double rsqrt_(double a) {
        const double r = (double)fast_rsqrt((float)a);
        return r * fma(-0.5 * a * r, r, 1.5);
    }
    static RM_HD double rcp_(double a) {
        const double r = (double)fast_div(1.f, (float)a);
        return r * fma(-a, r, 2.);
    }
    static RM_HD double sqrt_(double a) { return a > 0. ? a * rsqrt_(a) : 0.; }
    static RM_HD Vec3<double> normalized(Vec3<double> a);
};

template <typename R> RM_HD Vec3<R> operator+(Vec3<R> a, Vec3<R> b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
template <typename R> RM_HD Vec3<R> operator-(Vec3<R> a, Vec3<R> b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
template <typename R> RM_HD Vec3<R> operator*(Vec3<R> a, Vec3<R> b) { return {a.x * b.x, a.y * b.y, a.z * b.z}; }
template <typename R> RM_HD Vec3<R> operator-(Vec3<R> a) { return {-a.x, -a.y, -a.z}; }
template <typename R> RM_HD Vec3<R> scaled(Vec3<R> a, R s) { return {a.x * s, a.y * s, a.z * s}; }

// geometry.rs:180-182: v1.x*v2.x + v1.y*v2.y + v1.z*v2.z, left to right
template <typename R> RM_HD R dot(Vec3<R> a, Vec3<R> b) {
    return Num<R>::madd(a.z, b.z, Num<R>::madd(a.y, b.y, a.x * b.x));
}
template <> RM_HD double dot<double>(Vec3<double> a, Vec3<double> b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

template <typename R> RM_HD R squared_norm(Vec3<R> a) { return dot(a, a); }

// a + b*s  (e.g. orig + dir.scaled(t), sphere.rs:54)
template <typename R> RM_HD Vec3<R> axpy(Vec3<R> a, Vec3<R> b, R s) {
    return {Num<R>::madd(b.x, s, a.x), Num<R>::madd(b.y, s, a.y), Num<R>::madd(b.z, s, a.z)};
}
// a - b*s
template <typename R> RM_HD Vec3<R> axmy(Vec3<R> a, Vec3<R> b, R s) {
    return {Num<R>::nmadd(b.x, s, a.x), Num<R>::nmadd(b.y, s, a.y), Num<R>::nmadd(b.z, s, a.z)};
}

// geometry.rs:104-109: norm = sqrt(dot); if norm > 0 { scale(1/norm) }
template <typename R> RM_HD Vec3<R> normalized(Vec3<R> a) {
    R norm = Num<R>::sqrt_(dot(a, a));
    if (norm > R(0)) a = scaled(a, Num<R>::rcp_(norm));
    return a;
}

// f32: scale by rsqrt(|a|^2) -- one MUFU + Newton step instead of IEEE sqrt and reciprocal
template <> RM_HD Vec3<float> normalized<float>(Vec3<float> a) {
    const float s = dot(a, a);
    if (s > 0.f) a = scaled(a, fast_rsqrt(s));
    return a;
}

RM_HD Vec3<double> Fast64::normalized(Vec3<double> a) {
    const double s = a.x * a.x + a.y * a.y + a.z * a.z;
    if (s > 0.) a = scaled(a, rsqrt_(s));
    return a;
}
// numeric policies of the optics (rm_trace.cuh): Num<R> with the reference's normalisation, or Fast64
template <typename R> struct Exact : Num<R> {
    static RM_HD Vec3<R> normalized(Vec3<R> a) { return rm::normalized(a); }
};

// Keeps a value in its register across the code that follows: ptxas otherwise rematerialises cheap loop
// invariants (selects, offsets, int->float conversions) inside inner loops when registers are tight.
#if defined(__CUDA_ARCH__)
RM_HD void pin(float& v) { asm volatile("" : "+f"(v)); }
RM_HD void pin(double& v) { asm volatile("" : "+d"(v)); }
RM_HD void pin(int& v) { asm volatile("" : "+r"(v)); }
#else
RM_HD void pin(float&) {}
RM_HD void pin(double&) {}
RM_HD void pin(int&) {}
#endif
template <typename R> RM_HD void pin(Vec3<R>& v) { pin(v.x); pin(v.y); pin(v.z); }

template <typename R> RM_HD Vec3<R> xyz(const R4<R>& v) { return {v.x, v.y, v.z}; }

// Supersampled anti-aliasing (rm_render_supersampled): one output pixel as the mean of its S x S sub-pixels.
// sub_row(i, r) fills r[3 j + c] with channel c of sub-pixel j of sub-row i.  The order is normative (include/rm_b200.h):
// sub-rows outer, sub-pixels inner, FP32 adds without contraction (-fmad=false), then one IEEE division by S*S.  Sub-rows
// are handed over one at a time: a kernel need not hold all 3 S^2 values at once (S = 8: 192 floats).
template <int S, typename SubRow> RM_HD void resolve_box(const SubRow& sub_row, float out[3]) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
    for (int i = 0; i < S; i++) {
        float r[3 * S];
        sub_row(i, r);
#pragma unroll
        for (int j = 0; j < S; j++) {
            a0 += r[3 * j];
            a1 += r[3 * j + 1];
            a2 += r[3 * j + 2];
        }
    }
    const float n = (float)(S * S);
    out[0] = a0 / n;
    out[1] = a1 / n;
    out[2] = a2 / n;
}

// Adaptive anti-aliasing (rm_render_adaptive): whether pixel (x, y) of the 1x frame is refined (supersampled).  rgb (3
// floats per pixel) and id hold the frame's rows [lo, hi), row lo first, rows of `width` pixels; the caller makes [lo, hi)
// cover every row of [0, R) (R: the rendered rows) that the 3x3 neighbourhood of (x, y) reaches, and nothing beyond R.
// Normative (include/rm_b200.h): refined when `all`, or when one of the 8 neighbours inside [0, width) x [lo, hi) has
// another primitive id, or differs in some channel by more than k times the two values' sum -- Mitchell's contrast test,
// fabsf(a - b) > k * (a + b), FP32 without contraction.  k = +inf refines geometric edges only (inf * 0 is NaN).
RM_HD bool adaptive_mark(const float* rgb, const int* id, const int width, const int lo, const int hi, const int x, const int y,
                         const float k, const bool all) {
    if (all) return true;
    const size_t p = (size_t)(y - lo) * width + x;
    const int ip = id[p];
    const float a0 = rgb[3 * p], a1 = rgb[3 * p + 1], a2 = rgb[3 * p + 2];
    for (int dy = -1; dy <= 1; dy++) {
        const int qy = y + dy;
        if (qy < lo || qy >= hi) continue;
        for (int dx = -1; dx <= 1; dx++) {
            const int qx = x + dx;
            if ((dx == 0 && dy == 0) || qx < 0 || qx >= width) continue;
            const size_t q = (size_t)(qy - lo) * width + qx;
            if (id[q] != ip) return true;
            const float b0 = rgb[3 * q], b1 = rgb[3 * q + 1], b2 = rgb[3 * q + 2];
            if (fabsf(a0 - b0) > k * (a0 + b0) || fabsf(a1 - b1) > k * (a1 + b1) || fabsf(a2 - b2) > k * (a2 + b2)) return true;
        }
    }
    return false;
}

}  // namespace rm
