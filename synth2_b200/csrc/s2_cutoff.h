// s2_cutoff.h — filter coefficients of a MOVING cutoff, as a pure function of (voice parameters, frame offset).
//
// While the mod envelope ramps, the reference re-derives the filter coefficients every frame from
// fl = 2^(m * amount) * cutoff (process.rs:146-152, 231-250; filters.rs:17-21; dsp_filters.rs:99-109).  Round 1
// evaluated 2^x, sin and cos in binary64 per frame (~150 instructions); this file is the cheap form that still gives
// the reference's BITS in all but a percent of the frames — which matters: at low cutoffs the second-order
// low-pass's alpha = (1/2 + beta - gamma) / 4 cancels to 1e-5 and scatters by 1e-3 of itself from frame to frame
// with the last bit of cos, so two renders whose coefficients differ in most frames drift apart by several 1e-4
// (measured with a 2-ulp 2^x: 1 % of random banks outside the north-star bar), while rare one-ulp events do not.
//
//   * frame offsets are cut into absolute windows of 32 frames [32k, 32k + 32).  The window's centre frame gets the
//     binary64 evaluation (s2_math.h) of 2^x and of sin / cos of its angle, kept as hi + lo binary32 pairs;
//   * 2^x of a frame, x = RN(m * amount) exactly as the reference rounds it: 2^xc * 2^(x - xc), the second factor a
//     degree-4 polynomial in binary32 (|x - xc| <= 2^-5): correctly rounded but for ~0.1 % of arguments;
//   * fl = RN(2^x * cutoff) and theta = RN(RN(2 pi fl) / sr): the reference's own operations; the division by the
//     launch constant sr as q = a * (1/sr) plus one residual step (Markstein): the IEEE quotient for every a at the
//     usual rates (tools/check_cutoff.cpp checks 8 / 16 / 22.05 / 32 / 44.1 / 48 / 88.2 / 96 / 192 kHz exhaustively),
//     within an ulp for any other rate;
//   * sin / cos of a frame: the angle-addition correction in binary32 around the centre,
//     sin(tc + d) = S + (C sin d - S (1 - cos d)), |d| <= 2^-7 so sin d = d - d^3/6 and 1 - cos d = d^2/2 to 2e-10:
//     <= 1e-9 beyond a correct rounding (the rounded-once value in 99.5 % of the frames; glibc's own sinf / cosf,
//     which the oracle calls, differ from it in 1.3 %);
//   * the second-order coefficients from (sin, cos): the reference's own binary32 operations, one rounding each;
//     its num / den as reciprocal estimate, quotient, one residual correction (the IEEE quotient but for 1e-7 of
//     operands), so the scalar and the packed (two frames per instruction) forms are the same operations and give
//     the same bits.
//   * one-pole k = e^-theta: binary32 throughout (2^x by ex2.approx, the product theta * log2 e in two parts).
//     k only sets the cutoff — the filter's DC gain is (1-k)/(1-k) — so 2-3 ulp of k are far below the bar.
//
// PURITY.  Which evaluation a frame gets depends only on the voice's parameters and the frame's absolute offset
// (window index, envelope segment), never on how a render was cut into calls or chunks: a window is "valid" iff
// it lies inside one envelope segment, its centre angle times the segment's sweep rate stays below 2^-7 and the
// exponent moves by less than 2^-5 across half of it; frames of other windows get the full evaluation.  Every path of
// the kernels (moving-cutoff chunks packed and scalar, the general per-frame path, the time-split kernels) calls the
// functions below, so test_split_invariance_bitwise and test_paths_agree_bitwise keep holding.
//
// Host-and-device: tools/check_cutoff.cpp runs the scalar forms on the CPU.
#pragma once

#include "s2_math.h"

#ifdef __CUDACC__
#define S2C_FN __host__ __device__ __forceinline__
#else
#define S2C_FN inline
#endif

#ifdef __CUDA_ARCH__
#define S2C_ADD(a, b) __fadd_rn((a), (b))
#define S2C_MUL(a, b) __fmul_rn((a), (b))
#define S2C_FMA(a, b, c) __fmaf_rn((a), (b), (c))
#define S2C_DIV(a, b) __fdiv_rn((a), (b))
#else
#define S2C_ADD(a, b) ((a) + (b))
#define S2C_MUL(a, b) ((a) * (b))
#define S2C_FMA(a, b, c) fmaf((a), (b), (c))
#define S2C_DIV(a, b) ((a) / (b))
#endif

namespace s2c {

// ---- lane-vector operations: T = float (one frame) or float2 (frames i, i + 1 of one voice, device only) ----

S2C_FN float vadd(float a, float b) { return S2C_ADD(a, b); }
S2C_FN float vmul(float a, float b) { return S2C_MUL(a, b); }
S2C_FN float vfma(float a, float b, float c) { return S2C_FMA(a, b, c); }
S2C_FN float vmin(float a, float b) { return fminf(a, b); }
template <class T> struct Splat;
template <> struct Splat<float> { static S2C_FN float of(float x) { return x; } };
template <class T> S2C_FN T splat(float x) { return Splat<T>::of(x); }

// 2^x and 1/x by the special-function unit.  On the host (accuracy checks only) libm stands in.
S2C_FN float vex2(float x) {
#ifdef __CUDA_ARCH__
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return exp2f(x);
#endif
}
S2C_FN float vrcp(float x) {
#ifdef __CUDA_ARCH__
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
#else
    return 1.0f / x;
#endif
}

#ifdef __CUDACC__
// Blackwell packed-FP32 (FADD2 / FMUL2 / FFMA2): two IEEE results per issue slot, element-wise rounding.
// CONTRACTION HAZARD (ptxas 12.9): mul.rn.f32x2 feeding add.rn.f32x2 is fused into FFMA2 whatever the flags
// (tools/ubench/fuse_check.cu).  Rule: a packed product never feeds vadd; where the reference adds to a
// rounded product the add is vaddp(prod, y, one) = fma(prod, 1, y) with the 1 coming from a kernel
// parameter, which ptxas can neither fold nor fuse (there is no multiply-multiply-add) — same bits as an add.
#ifndef S2_SCALAR_PAIRS
__device__ __forceinline__ float2 vadd(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "add.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 vmul(float2 a, float2 b) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
        "mul.rn.f32x2 rd, ra, rb;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 vfma(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
#else   // experiment: the same element-wise operations as two scalar instructions (same bits)
__device__ __forceinline__ float2 vadd(float2 a, float2 b) { return make_float2(__fadd_rn(a.x, b.x), __fadd_rn(a.y, b.y)); }
__device__ __forceinline__ float2 vmul(float2 a, float2 b) { return make_float2(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)); }
__device__ __forceinline__ float2 vfma(float2 a, float2 b, float2 c) { return make_float2(__fmaf_rn(a.x, b.x, c.x), __fmaf_rn(a.y, b.y, c.y)); }
#endif
template <> struct Splat<float2> { static __device__ __forceinline__ float2 of(float x) { return make_float2(x, x); } };
__device__ __forceinline__ float2 vex2(float2 x) { return make_float2(vex2(x.x), vex2(x.y)); }
__device__ __forceinline__ float2 vrcp(float2 x) { return make_float2(vrcp(x.x), vrcp(x.y)); }
__device__ __forceinline__ float2 vmin(float2 a, float b) { return make_float2(fminf(a.x, b), fminf(a.y, b)); }
#endif

// prod + y with its own rounding, where prod may come from a packed multiply (see the hazard note)
template <class T> S2C_FN T vaddp(T prod, T y, float one) { return vfma(prod, splat<T>(one), y); }

// ---- the per-frame chain ----

constexpr float kTwoPi = 6.28318548202636718750f;      // 2.0 * std::f32::consts::PI in binary32 (filters.rs:21)
constexpr float kWinDelta = 0.0078125f;                // 2^-7: the largest |theta - theta_c| a valid window allows
constexpr float kWinDeltaX = 0.03125f;                 // 2^-5: the largest |x - x_c| (exponent of 2^x)
constexpr uint32_t kWinShift = 5;                      // windows of 32 frames
constexpr float kThetaMax = 3.125f;                    // a valid window's centre angle: theta stays below pi

// theta = (2 pi fl) / sr (dsp_filters.rs:107, filters.rs:21 with the sign dropped).  rsr = RN(1 / sr).
template <class T>
S2C_FN T theta_of(T fl, float sr, float rsr) {
    const T a = vmul(fl, splat<T>(kTwoPi));
    const T q = vmul(a, splat<T>(rsr));
    const T e = vfma(splat<T>(-sr), q, a);             // exact residual a - sr q
    return vfma(e, splat<T>(rsr), q);
}

// theta of the one-pole's moving cutoff: 2^(m * amount) * theta0, theta0 = (2 pi cutoff) / sr, 2^x by the hardware
template <class T>
S2C_FN T theta_at(T m, float amount, float theta0) { return vmul(vex2(vmul(m, splat<T>(amount))), splat<T>(theta0)); }

// num / den for den in [1, 9], |num| <= 8: reciprocal estimate, quotient, one residual correction.  nden = -den.
template <class T>
S2C_FN T div_in_range_from(T num, T nden, T r) {        // r ~ 1 / den to within 2 ulp
    const T q = vmul(num, r);
    return vfma(vfma(nden, q, num), r, q);
}
template <class T>
S2C_FN T div_in_range(T num, T den, T nden) { return div_in_range_from(num, nden, vrcp(den)); }

// k = e^-theta in binary32 (one-pole, filters.rs:21): 2^-(theta log2 e), log2 e = L1 + L2, the product in two parts:
// tn = RN(theta * -L1), r = theta * L1 + tn (exact), tl = r + theta * L2, k = 2^tn * (1 - tl ln 2).
// theta is first clamped to kThetaBig: a cutoff modulated past binary32 (2^(m amount) with m amount >= 128, or
// 2 pi f beyond the largest float) gives theta = +inf, and then r = inf - inf is NaN where the reference's
// exp(-inf) is 0.  Below the clamp nothing changes; from it up to ~2.3e38 the result was already 0 (2^tn
// underflows), and above that theta * L1 overflows and the unclamped form gave NaN too.
constexpr float kThetaBig = 128.0f;
template <class T>
S2C_FN T exp_neg_fast(T th) {
    const float L1 = 0x1.715476p+0f, L2 = 0x1.4ae0c0p-26f;
    th = vmin(th, kThetaBig);
    const T tn = vmul(th, splat<T>(-L1));
    const T r = vfma(th, splat<T>(L1), tn);
    const T tl = vfma(th, splat<T>(L2), r);
    const T e = vex2(tn);
    return vfma(e, vmul(tl, splat<T>(-0x1.62e430p-1f)), e);
}

// The centre of one 32-frame window of a cutoff trajectory: the exponent and the angle of its centre frame and the
// binary64 values of 2^x, sin and cos there, as hi + lo binary32 pairs.  valid = 0: frames of this window take the
// full evaluation.
struct Window {
    uint32_t k;             // window index (frame offset >> 5); 0xffffffff = none yet
    uint32_t valid;
    float xc;               // RN(m * amount) of the centre frame
    float Eh, Er;           // 2^xc = Eh (1 + Er)
    float thc;              // theta of the centre frame, through the reference's chain from RN(2^xc)
    float Ah, Al, Bh, Bl;   // sin (A) and cos (B) of thc
};

S2C_FN void split_hi_lo(double v, float* hi, float* lo) {
    *hi = (float)v;
    *lo = (float)(v - (double)*hi);
}
// v = hi (1 + rel), |rel| <= 2^-24 known to ~2^-24 of itself
S2C_FN void split_hi_rel(double v, float* hi, float* rel) {
    float lo;
    split_hi_lo(v, hi, &lo);
    *rel = S2C_DIV(lo, *hi);
}

// sin(thc + d), cos(thc + d) from the window (|d| <= 2^-7):
// S + (C sin d - S (1 - cos d)) and C - (S sin d + C (1 - cos d)), the low parts of S and C folded into the
// second-order terms.
template <class T>
S2C_FN void window_sincos(const Window& W, T d, T* s, T* c) {
    const T z = vmul(d, d);
    const T sd = vfma(vmul(d, z), splat<T>(-0x1.555556p-3f), d);          // sin d = d - d^3 / 6
    const T ws = vfma(splat<T>(-0.5f * W.Ah), z, splat<T>(W.Al));         // Al - S d^2 / 2
    *s = vadd(splat<T>(W.Ah), vfma(splat<T>(W.Bh), sd, ws));
    const T wc = vfma(splat<T>(-0.5f * W.Bh), z, splat<T>(W.Bl));         // Bl - C d^2 / 2
    *c = vadd(splat<T>(W.Bh), vfma(splat<T>(-W.Ah), sd, wc));
}

// 2^x for x = RN(m * amount) inside the window (|x - xc| <= 2^-5): 2^xc * 2^d = Eh (1 + Er + (2^d - 1)),
// 2^d - 1 = d (L + d (L^2/2 + d (L^3/6 + d L^4/24))), L = ln 2.  x is a rounded product and must stay one: the
// difference is taken through an fma by an opaque 1 (see the hazard note), in the scalar form too, so both are the
// same operations.
template <class T>
S2C_FN T sweep_exact(const Window& W, T x, float one) {
    const T d = vfma(x, splat<T>(one), splat<T>(-W.xc));                  // exact (Sterbenz) or far below an ulp of x
    T p = vfma(d, splat<T>(0x1.3b2ab6p-7f), splat<T>(0x1.c6b08ep-5f));    // L^4/24 d + L^3/6
    p = vfma(p, d, splat<T>(0x1.ebfbe0p-3f));                             // + L^2/2
    p = vfma(p, d, splat<T>(0x1.62e430p-1f));                             // + L
    const T em = vfma(d, p, splat<T>(W.Er));
    return vfma(splat<T>(W.Eh), em, splat<T>(W.Eh));
}

// q = (1 - h) / (1 + h), h = hd * sin (dsp_filters.rs:108 / :158 with beta = q / 2), for 1 <= 1 + h <= 9
template <class T>
S2C_FN T quotient_of(T s, float hd, float one) {
    const T h = vmul(splat<T>(hd), s);
    const T num = vfma(h, splat<T>(-one), splat<T>(1.0f));               // 1 - h, one rounding (exact product)
    const T den = vfma(h, splat<T>(one), splat<T>(1.0f));                // 1 + h
    const T nden = vfma(h, splat<T>(-one), splat<T>(-1.0f));             // -(1 + h): the same rounding, mirrored
    return div_in_range(num, den, nden);
}

// Second-order low-pass / high-pass coefficients from q and cos (dsp_filters.rs:99-109, :149-159), with the output
// doubling folded in: c0 = 2 alpha, c1 = 2 beta, c2 = 2 gamma.  Scaling by a power of two commutes with
// round-to-nearest, so with q = 2 beta: 1/2 + beta = RN(1 + q) / 2, 2 gamma = RN(RN(1 + q) cos),
// 2 alpha = RN(RN(1 + q) -+ 2 gamma) / 4 — the reference's roundings, fewer operations.
template <bool HIGH_PASS, class T>
S2C_FN void biquad_from_q_cos(T q, T co, float one, T* c0, T* c1, T* c2) {
    const T hb2 = vadd(q, splat<T>(1.0f));
    const T g2 = vmul(hb2, co);
    const T t = vfma(g2, splat<T>(HIGH_PASS ? one : -one), hb2);           // RN(hb2 -+ g2)
    *c0 = vmul(t, splat<T>(0.25f));
    *c1 = q;
    *c2 = g2;
}

// From sin and cos.  Callers guarantee 1 <= 1 + h <= 9 (a valid window: 0 < theta < pi and 0 <= hd <= 8); anything
// else goes through biquad_lp_hp_any below.  hd = damping / 2.
template <bool HIGH_PASS, class T>
S2C_FN void biquad_lp_hp(T s, T co, float hd, float one, T* c0, T* c1, T* c2) {
    biquad_from_q_cos<HIGH_PASS, T>(quotient_of<T>(s, hd, one), co, one, c0, c1, c2);
}

// The same coefficients for any operands (frames outside valid windows): inside the straight-line division's
// range (every stable filter: 0 < theta < pi, damping in [0, 16]) it IS biquad_lp_hp; outside it the division is
// the IEEE one.
template <bool HIGH_PASS>
S2C_FN void biquad_lp_hp_any(float s, float co, float hd, float one, float* c0, float* c1, float* c2) {
    const float h = vmul(hd, s);
    const float den = vfma(h, one, 1.0f);
    if (den >= 1.0f && den <= 9.0f) {
        biquad_lp_hp<HIGH_PASS, float>(s, co, hd, one, c0, c1, c2);
        return;
    }
    const float num = vfma(h, -one, 1.0f);
    const float q = S2C_DIV(num, den);
    const float hb2 = vadd(q, 1.0f);
    const float g2 = vmul(hb2, co);
    const float t = vfma(g2, HIGH_PASS ? one : -one, hb2);
    *c0 = vmul(t, 0.25f);
    *c1 = q;
    *c2 = g2;
}

}  // namespace s2c
