// s2_device.cuh — device-side building blocks shared by the render kernels (s2_kernels.cu: one warp per
// 32 voices; s2_kernel_ts.cu: one warp per voice, lanes = time segments).
//
// Arithmetic contract: every operation below that feeds a discrete decision (phase, table index,
// envelope stage, noise hash) is the reference's binary32 operation, spelled with __f*_rn intrinsics so
// nothing is contracted or reassociated (the files are also built with -fmad=false).
// Reference line numbers are relative to /root/reference/components/s2_lib/src/.
#pragma once

#include "s2_internal.h"
#include "s2_math.h"
#include "s2_cutoff.h"

#include <type_traits>

// The biquad's products and sums are rounded separately, as the source reads (dsp_filters.rs:116-128).  A
// fused (FFMA) form was tried and rejected: a resonant low-cutoff biquad in f32 direct form amplifies
// per-frame rounding differences by ~1/(1-r) (~10^3 at 100 Hz, damping 0.2), enough to pass the 1e-4 bar.
// (The fast phase step was also tried as a separate pass ahead of everything else: slower, row d of
// profiles/r1_notes.md.)

// Frames per straight-line trip of the time-packed loop; 16 and 32 measured no faster than 8.
#ifndef S2_TRIP
#define S2_TRIP 8
#endif

namespace s2 {


static __device__ const uint32_t d_sin_bits[1024] = {
#include "sin_table_bits.inc"
};

// Oscillator-kind dispatch: fn(std::integral_constant<int, K>, args...) for the first K of the list equal to k, the
// last K of the list for any other k.  The list is the set of loop variants a call site instantiates.  The loop's
// arguments are passed through rather than captured: a lambda that captures the render kernel's locals by reference
// changes its register allocation (e.g. 8 B of spills appear or vanish, instruction counts move by up to 5 %).
template <int K, int... Ks, class Fn, class... A>
__device__ __forceinline__ void with_kind(int k, Fn&& fn, A&&... args) {
    if constexpr (sizeof...(Ks) == 0) fn(std::integral_constant<int, K>{}, args...);
    else if (k == K) fn(std::integral_constant<int, K>{}, args...);
    else with_kind<Ks...>(k, fn, args...);
}

// ------------------------------------------------------------------------------------------
// Per-lane voice description, decoded once per launch.

struct EnvP {
    float A, AD, S, Rs, E;   // stage boundaries in samples: attack end, decay end, release start/end
    float D, R;              // decay / release lengths in samples (scalar tail path)
    float relf;              // release_offset as f32 (None -> u32::MAX as f32), before the max()
    float sA, sD, sR;        // hoisted slopes rise/run of the x16 envelope (old/simdtest.rs:247-251)
};

struct OscC {                // everything derived from the period; hoisting a division whose
    float P, d;              // operands do not change is exact
    float slope;             // -2 / P            (saw,      try3/oscillators.rs:99-119)
    float half;              // P / 2             (square,   try3/oscillators.rs:60-80)
    float ts1, ts2;          // -2 / half, 2 / half (triangle, try3/oscillators.rs:148-183)
    uint32_t fo_bits;        // frequency these were derived from
};

struct FiltC {               // one-pole: c0 = k, c1 = 1 - k.   biquad: c0 = 2*alpha, c1 = 2*beta, c2 = 2*gamma
    float c0, c1, c2;
    uint32_t fl_bits;
};

struct FiltS { float x1, x2, y1, y2; };   // one-pole keeps `last` in y1

struct Lane {
    uint32_t kind, rot;      // rot = seed.rotate_left(5)  (try3/hashnoise.rs:53-55)
    float pitch, gain, namt, lpf, damp, amt_osc, amt_lpf;
    EnvP amp, mod;
};

// units.rs:44-53
__device__ __forceinline__ float ms_as_samples(float ms, float sr) {
    return __fmul_rn(sr, __fdiv_rn(ms, 1000.0f));
}

__device__ __forceinline__ void make_env(EnvP& e, float a_ms, float d_ms, float s, float r_ms,
                                         uint32_t release, float sr) {
    e.A = ms_as_samples(a_ms, sr);
    e.D = ms_as_samples(d_ms, sr);
    e.R = ms_as_samples(r_ms, sr);
    e.S = s;
    e.AD = __fadd_rn(e.A, e.D);
    e.relf = __uint2float_rn(release);             // unwrap_or(u32::MAX) as f32 (simdtest.rs:283)
    e.Rs = fmaxf(e.relf, e.AD);                    // simd_max (simdtest.rs:285)
    e.E = __fadd_rn(e.Rs, e.R);
    e.sA = __fdiv_rn(1.0f, e.A);
    e.sD = __fdiv_rn(__fsub_rn(s, 1.0f), e.D);
    e.sR = __fdiv_rn(-s, e.R);
}

// old/simdtest.rs:287-291: the mask chain, as a stage index
template <class E>
__device__ __forceinline__ int env_stage(const E& e, float x) {
    return x < e.A ? 0 : (x < e.AD ? 1 : (x < e.Rs ? 2 : (x < e.E ? 3 : 4)));
}

// old/simdtest.rs:270-330 for one lane; line = (rise/run)*x + y0, never fused (:247-261)
template <class E>
__device__ __forceinline__ float env_x16(const E& e, float x) {
    switch (env_stage(e, x)) {
    case 0: return __fadd_rn(__fmul_rn(e.sA, x), 0.0f);
    case 1: return __fadd_rn(__fmul_rn(e.sD, __fsub_rn(x, e.A)), 1.0f);
    case 2: return e.S;
    case 3: return __fadd_rn(__fmul_rn(e.sR, __fsub_rn(x, e.Rs)), e.S);
    default: return 0.0f;
    }
}

// The envelope segment a frame offset lies in, as the line g = es * (x - ex0) + ey0 that reproduces that
// stage's formula bit-for-bit (attack: (1/A)*x + 0; decay: ((S-1)/D)*(x-A) + 1; sustain: 0*x + S; release:
// ((-S)/R)*(x-Rs) + S; end: 0*x + 0), valid for frame offsets [.., nend).  Offsets below 2^24 only
// (x = (f32)n exact; nend = first integer whose f32 image reaches the stage boundary).
struct SegEnv { float es, nex0, ey0; uint32_t nbeg, nend; int stage; };

// first integer frame offset whose f32 image reaches the boundary b (exact below 2^24)
__device__ __forceinline__ uint32_t env_bound(float b) { return min(__float2uint_ru(b), 1u << 24); }

template <class E>
__device__ __forceinline__ SegEnv seg_env(const E& e, uint32_t n) {
    const float x = __uint2float_rn(n);
    const int st = env_stage(e, x);
    SegEnv s;
    s.stage = st;
    s.es = st == 0 ? e.sA : st == 1 ? e.sD : st == 3 ? e.sR : 0.0f;
    s.nex0 = st == 1 ? -e.A : st == 3 ? -e.Rs : -0.0f;             // x + (-0.0) == x
    s.ey0 = st == 1 ? 1.0f : (st == 2 || st == 3) ? e.S : 0.0f;
    const float b = st == 0 ? e.A : st == 1 ? e.AD : st == 2 ? e.Rs : st == 3 ? e.E : 4.0e9f;
    const float a = st == 0 ? 0.0f : st == 1 ? e.A : st == 2 ? e.AD : st == 3 ? e.Rs : e.E;
    s.nend = env_bound(b);
    s.nbeg = env_bound(a);
    return s;
}
__device__ __forceinline__ float seg_eval(const SegEnv& s, float x) {
    return __fadd_rn(__fmul_rn(s.es, __fadd_rn(x, s.nex0)), s.ey0);
}
// The envelope at frame offset n (x = its f32 image) of a walk that keeps its current segment in `s`: the line inside
// the segment, the stage chain at a boundary, after which `s` is the next frame's segment.
template <class E>
__device__ __forceinline__ float seg_walk(SegEnv& s, const E& e, uint32_t n, float x) {
    if (n < s.nend) return seg_eval(s, x);
    const float g = env_x16(e, x);
    s = seg_env(e, n + 1u);
    return g;
}

// fmod(t, 1) for t in [0, 2) (the fast paths: 0 <= phase < 1, 0 <= 1/P < 1): t - 1 is exact there, and as
// unsigned integers the bits of a negative t - 1 exceed those of any t < 1 while a non-negative t - 1 lies
// below t >= 1, so the wrap is one integer min.  No predicate: FSETP/ISETP -> FSEL or a predicated FADD costs
// 14 cycles of latency on this part against 6.75 for VIMNMX (tools/ubench/phase_chain.cu: 22.9 -> 14.75 cycles
// per step of the recurrence, same bits).
__device__ __forceinline__ float wrap_unit(float t) {
    return __uint_as_float(min(__float_as_uint(__fadd_rn(t, -1.0f)), __float_as_uint(t)));
}

// math.rs:11-19 with feature "fma"
__device__ __forceinline__ float line_fma(float rise, float run, float x, float y0) {
    return __fmaf_rn(__fdiv_rn(rise, run), x, y0);
}

// try3/envelopes.rs:22-149 (tail frames only)
__device__ __forceinline__ float env_scalar(const EnvP& e, float x) {
    const float rel = e.relf;
    const float end = __fadd_rn(rel, e.R);
    const bool in_release = x >= rel && x < end;
    const bool in_end = x >= end;
    const bool in_attack = !in_release && !in_end && x < e.A;
    const bool in_decay = !in_release && !in_end && !in_attack && x < e.AD;
    const bool in_sustain = !in_release && !in_end && !in_attack && !in_decay && x < rel;
    float rss;
    if (rel < e.A) rss = line_fma(1.0f, e.A, rel, 0.0f);
    else if (rel < e.AD) rss = line_fma(__fsub_rn(e.S, 1.0f), e.D, __fsub_rn(rel, e.A), 1.0f);
    else rss = e.S;
    if (in_attack) return line_fma(1.0f, e.A, x, 0.0f);
    if (in_decay) return line_fma(__fsub_rn(e.S, 1.0f), e.D, __fsub_rn(x, e.A), 1.0f);
    if (in_sustain) return e.S;
    if (in_release) return line_fma(-rss, e.R, __fsub_rn(x, rel), rss);
    return 0.0f;
}

// 2^x, e^x, sin/cos: s2_math.h (binary64 evaluation, one rounding).  The reference calls sleef pow
// (x16, process.rs:244) / libm powf (scalar, process.rs:227) / expf / sinf / cosf, none reproducible
// bit-for-bit on a GPU; their outputs only feed float results, compared with the north-star tolerance.
__device__ __forceinline__ float pow2_ref(float x) { return s2_exp2f(x); }
__device__ __forceinline__ float exp_ref(float x) { return s2_expf(x); }

// process.rs:231-250.  amount == 0 -> pow(2, +-0) == 1 and 1 * f == f exactly: skip the call.
__device__ __forceinline__ float modulate_freq(float f, float m, float amount) {
    if (amount == 0.0f) return f;
    return __fmul_rn(pow2_ref(__fmul_rn(m, amount)), f);
}

__device__ __forceinline__ void make_osc(OscC& o, float fo, float sr) {
    o.fo_bits = __float_as_uint(fo);
    o.P = __fdiv_rn(sr, fo);                       // units.rs:32-41
    o.d = __fdiv_rn(1.0f, o.P);                    // try3/oscillators.rs:378
    o.slope = __fdiv_rn(-2.0f, o.P);
    o.half = __fdiv_rn(o.P, 2.0f);
    o.ts1 = __fdiv_rn(-2.0f, o.half);
    o.ts2 = __fdiv_rn(2.0f, o.half);
}

// FILTER template values = S2_FILTER_* of include/s2_cuda.h
enum { FILT_ONE_POLE = 0, FILT_BIQUAD_LP = 1, FILT_BIQUAD_HP = 2, FILT_BIQUAD_BP = 3, FILT_FIRST_LP = 4, FILT_FIRST_HP = 5 };

// theta = (2 pi f) / sr: try3/filters.rs:21 with the sign dropped, dsp_filters.rs:107
__device__ __forceinline__ float theta_ref(float fl, float sr) {
    const float pi = 3.14159274101257324219f;
    return __fdiv_rn(__fmul_rn(__fmul_rn(2.0f, pi), fl), sr);
}

// Coefficients of every filter but the one-pole from theta, all transcendentals in binary64 rounded once
template <int FILTER>
__device__ __forceinline__ void make_filt_theta(FiltC& c, float th, float damp) {
    if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP) {
        // try3/dsp_filters.rs:99-109 (low-pass), :149-159 (high-pass: alpha = (1/2 + beta + gamma) / 4)
        float s, co;
        s2_sincosf(th, &s, &co);
        const float hd = __fmul_rn(damp, 0.5f);                      // damp / 2.0: scaling by a power of two, same bits
        const float num = __fsub_rn(1.0f, __fmul_rn(hd, s));
        const float den = __fadd_rn(1.0f, __fmul_rn(hd, s));
        const float beta = __fmul_rn(0.5f, __fdiv_rn(num, den));
        const float gamma = __fmul_rn(__fadd_rn(0.5f, beta), co);
        const float hb = __fadd_rn(0.5f, beta);
        const float alpha = __fmul_rn(FILTER == FILT_BIQUAD_LP ? __fsub_rn(hb, gamma) : __fadd_rn(hb, gamma), 0.25f);   // ... / 4.0, likewise
        // y = 2*(alpha*s + gamma*y1 - beta*y2): scaling by 2 commutes with round-to-nearest, so the
        // doubling is folded into the coefficients (exact unless an intermediate is subnormal).
        c.c0 = __fmul_rn(2.0f, alpha);
        c.c1 = __fmul_rn(2.0f, beta);
        c.c2 = __fmul_rn(2.0f, gamma);
    } else if (FILTER == FILT_BIQUAD_BP) {
        // try3/dsp_filters.rs:197-207; `damp` carries the quality factor
        const float tn = s2_tanf(__fdiv_rn(th, __fmul_rn(2.0f, damp)));
        const float beta = __fmul_rn(0.5f, __fdiv_rn(__fsub_rn(1.0f, tn), __fadd_rn(1.0f, tn)));
        float s, co;
        s2_sincosf(th, &s, &co);
        const float gamma = __fmul_rn(__fadd_rn(0.5f, beta), co);
        const float alpha = __fmul_rn(__fsub_rn(0.5f, beta), 0.5f);
        c.c0 = __fmul_rn(2.0f, alpha);
        c.c1 = __fmul_rn(2.0f, beta);
        c.c2 = __fmul_rn(2.0f, gamma);
    } else {
        // try3/dsp_filters.rs:30-32 (first-order low-pass) / :64-66 (high-pass): c0 = alpha, c2 = gamma
        float s, co;
        s2_sincosf(th, &s, &co);
        const float gamma = __fdiv_rn(co, __fadd_rn(1.0f, s));
        c.c0 = __fmul_rn(FILTER == FILT_FIRST_LP ? __fsub_rn(1.0f, gamma) : __fadd_rn(1.0f, gamma), 0.5f);
        c.c1 = 0.0f;
        c.c2 = gamma;
    }
}

// Coefficients of a RESTING cutoff (every frame whose mod envelope is in sustain / end, or whose cutoff does not
// follow it; also the scalar tail): the reference's chain, transcendentals in binary64.
template <int FILTER>
__device__ __forceinline__ void make_filt(FiltC& c, float fl, float damp, float sr) {
    c.fl_bits = __float_as_uint(fl);
    if (FILTER == 0) {
        // try3/filters.rs:21: (-2.0 * pi * freq / sample_rate).exp()
        const float pi = 3.14159274101257324219f;
        float t = __fmul_rn(-2.0f, pi);
        t = __fmul_rn(t, fl);
        t = __fdiv_rn(t, sr);
        const float k = exp_ref(t);
        c.c0 = k;
        c.c1 = __fsub_rn(1.0f, k);
        c.c2 = 0.0f;
    } else {
        make_filt_theta<FILTER>(c, theta_ref(fl, sr), damp);
    }
}

// ------------------------------------------------------------------------------------------
// MOVING cutoff (s2_cutoff.h): the mod envelope is in a ramp (attack / decay / release) and the cutoff follows it.

struct CutP {            // per-voice constants of the moving evaluation
    float lpf;           // the patch's cutoff in Hz
    float theta0;        // (2 pi cutoff) / sr — the one-pole's form
    float amt;           // mod_env_to_lpf_freq
    float damp, hd;      // damping, damping / 2
    float sr, rsr;       // sample rate and RN(1 / sr)
};
__device__ __forceinline__ CutP cutp_of(float lpf, float theta0, float amt_lpf, float damp, float sr, float rsr) {
    CutP c;
    c.lpf = lpf;
    c.theta0 = theta0;
    c.amt = amt_lpf;
    c.damp = damp;
    c.hd = __fmul_rn(damp, 0.5f);
    c.sr = sr;
    c.rsr = rsr;
    return c;
}
__device__ __forceinline__ CutP make_cutp(float lpf, float amt_lpf, float damp, float sr) {
    return cutp_of(lpf, theta_ref(lpf, sr), amt_lpf, damp, sr, __frcp_rn(sr));
}

// theta of the frame whose mod envelope is m by the reference's own chain, 2^x in binary64 rounded once
// (process.rs:244-246, dsp_filters.rs:107): the evaluation of frames outside valid windows and of window centres.
__device__ __forceinline__ float theta_full(const CutP& cp, float m) {
    return theta_ref(__fmul_rn(s2_exp2f(__fmul_rn(m, cp.amt)), cp.lpf), cp.sr);
}

// The window of frame offset n inside mod-envelope segment sm (a ramp).  Valid iff the 32 frames of the window
// lie in the segment, the centre angle leaves room below pi, across half a window the exponent stays within 2^-5
// (it moves by amt * es per frame) and the angle within 2^-7 (|d| <= thc * 16 ln 2 |amt es| (1 + ...) < thc * 12 |amt es|)
// and the damping suits the straight-line division.  A pure function of (voice, n >> 5).
template <int FILTER>
__device__ __forceinline__ void make_window_inl(s2c::Window& W, const SegEnv& sm, const CutP& cp, uint32_t n) {
    const uint32_t k = n >> s2c::kWinShift;
    W.k = k;
    const uint32_t w0 = k << s2c::kWinShift;
    const float xc = __fmul_rn(seg_eval(sm, __uint2float_rn(w0 + 16u)), cp.amt);
    const float r = fabsf(__fmul_rn(cp.amt, sm.es));
    const float r12 = __fmul_rn(r, 12.0f);
    const bool in_range = xc > -100.0f && xc < 100.0f && __fmul_rn(r, 17.0f) <= s2c::kWinDeltaX;
    double Ed = 0.0;
    float thc = 4.0f;
    if (in_range) {
        Ed = s2_exp2_d(xc);
        thc = theta_ref(__fmul_rn((float)Ed, cp.lpf), cp.sr);
    }
    bool valid = in_range && w0 >= sm.nbeg && w0 + 32u <= sm.nend && thc <= s2c::kThetaMax &&
                 __fmul_rn(thc, r12) <= s2c::kWinDelta;
    if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP) valid = valid && cp.hd >= 0.0f && cp.hd <= 8.0f;
    if (FILTER == FILT_ONE_POLE || FILTER == FILT_BIQUAD_BP) valid = false;      // these never look at a window
    W.valid = valid ? 1u : 0u;
    W.xc = xc;
    W.thc = thc;
    if (valid) {
        double sd, cd;
        s2_sincos_d((double)thc, &sd, &cd);
        s2c::split_hi_rel(Ed, &W.Eh, &W.Er);
        s2c::split_hi_lo(sd, &W.Ah, &W.Al);
        s2c::split_hi_lo(cd, &W.Bh, &W.Bl);
    } else {
        W.Eh = W.Er = W.Ah = W.Al = W.Bh = W.Bl = 0.0f;
    }
}

__device__ __forceinline__ void window_none(s2c::Window& W) {
    W.k = 0xffffffffu; W.valid = 0u; W.xc = 0.0f; W.thc = 0.0f;
    W.Eh = W.Er = W.Ah = W.Al = W.Bh = W.Bl = 0.0f;
}

template <int FILTER>
__device__ __noinline__ void make_window(s2c::Window& W, const SegEnv& sm, const CutP& cp, uint32_t n) {
    make_window_inl<FILTER>(W, sm, cp, n);
}

// sin and cos of the angle of the frame(s) whose mod envelope is m, inside valid window W: the reference's chain
// in binary32 around the window's centre (s2_cutoff.h).  T = float or float2, the same operations.
template <class T>
__device__ __forceinline__ void window_frame_sincos(const s2c::Window& W, const CutP& cp, float one, T m, T* s, T* co) {
    const T E = s2c::sweep_exact<T>(W, s2c::vmul(m, s2c::splat<T>(cp.amt)), one);
    const T th = s2c::theta_of<T>(s2c::vmul(E, s2c::splat<T>(cp.lpf)), cp.sr, cp.rsr);
    s2c::window_sincos<T>(W, s2c::vadd(th, s2c::splat<T>(-W.thc)), s, co);
}

// Coefficients of one moving frame (scalar form): m = the mod envelope at frame n (inside segment sm).
template <int FILTER>
__device__ __forceinline__ void moving_coefs(FiltC& c, s2c::Window& W, const SegEnv& sm, const CutP& cp, float one,
                                             uint32_t n, float m) {
    c.fl_bits = kNoKey;                                   // not a memo of any resting cutoff
    if (FILTER == FILT_ONE_POLE) {
        const float k = s2c::exp_neg_fast<float>(s2c::theta_at<float>(m, cp.amt, cp.theta0));
        c.c0 = k;
        c.c1 = __fsub_rn(1.0f, k);
        c.c2 = 0.0f;
        return;
    }
    if (FILTER == FILT_BIQUAD_BP) { make_filt_theta<FILTER>(c, theta_full(cp, m), cp.damp); return; }
    if ((n >> s2c::kWinShift) != W.k) make_window<FILTER>(W, sm, cp, n);
    if (W.valid) {
        float s, co;
        window_frame_sincos<float>(W, cp, one, m, &s, &co);
        if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP) {
            s2c::biquad_lp_hp<FILTER == FILT_BIQUAD_HP, float>(s, co, cp.hd, one, &c.c0, &c.c1, &c.c2);
        } else {
            const float gamma = __fdiv_rn(co, __fadd_rn(1.0f, s));
            c.c0 = __fmul_rn(FILTER == FILT_FIRST_LP ? __fsub_rn(1.0f, gamma) : __fadd_rn(1.0f, gamma), 0.5f);
            c.c1 = 0.0f;
            c.c2 = gamma;
        }
    } else if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP) {
        float s, co;
        s2_sincosf(theta_full(cp, m), &s, &co);
        s2c::biquad_lp_hp_any<FILTER == FILT_BIQUAD_HP>(s, co, cp.hd, one, &c.c0, &c.c1, &c.c2);
    } else {
        make_filt_theta<FILTER>(c, theta_full(cp, m), cp.damp);
    }
}

// Does the cutoff of a voice move at x16 frame n?  (amount != 0 and the mod envelope is in a ramp)
__device__ __forceinline__ bool stage_moves(int stage) { return stage == 0 || stage == 1 || stage == 3; }

// The compact envelope the classifier and the per-frame evaluation need (env_stage / env_x16); the
// scalar-tail envelope (env_scalar) needs the full EnvP.
struct EnvQ { float A, AD, S, Rs, E, sA, sD, sR; };
__device__ __forceinline__ EnvQ compact(const EnvP& e) { return {e.A, e.AD, e.S, e.Rs, e.E, e.sA, e.sD, e.sR}; }

// Decode one voice's parameter column (struct-of-arrays, see s2_internal.h).
__device__ __forceinline__ Lane load_lane(const float* __restrict__ P, uint32_t vp, float sr, uint32_t release) {
    Lane L;
    L.kind = __float_as_uint(P[P_KIND * vp]);
    const uint32_t seed = __float_as_uint(P[P_SEED * vp]);
    L.rot = (seed << 5) | (seed >> 27);
    L.pitch = P[P_PITCH * vp];
    L.gain = P[P_GAIN * vp];
    L.namt = P[P_NOISE * vp];
    L.lpf = P[P_LPF * vp];
    L.damp = P[P_DAMP * vp];
    L.amt_osc = P[P_AMT_OSC * vp];
    L.amt_lpf = P[P_AMT_LPF * vp];
    make_env(L.amp, P[P_AA * vp], P[P_AD * vp], P[P_AS * vp], P[P_AR * vp], release, sr);
    make_env(L.mod, P[P_MA * vp], P[P_MD * vp], P[P_MS * vp], P[P_MR * vp], release, sr);
    return L;
}

// ------------------------------------------------------------------------------------------
// One frame of one voice.

// phased + basic oscillators (try3/oscillators.rs:217-239 then :60-199) and the phase step
// (:377-381).  LITERAL keeps both `%`; the fast form drops them where they are provably no-ops:
//   * RN(P * phase) < P for every phase < 1 (P - P*2^-24 lies more than half an ulp below P),
//     so `offset % period` returns its argument;
//   * phase + 1/P < 2 when 1/P < 1, so `% 1.0` is a conditional exact subtraction.
template <int KIND, bool LITERAL>
__device__ __forceinline__ float osc_step(uint32_t kind, const OscC& o, float& ph, const float* sintab) {
    float x = __fmul_rn(o.P, ph);                  // period.mul_add(phase, 0.0)
    if (LITERAL) x = fmodf(x, o.P);
    const uint32_t k = KIND >= 0 ? (uint32_t)KIND : kind;
    float y;
    if (k == 1u) {                                 // Saw
        y = __fmaf_rn(o.slope, x, 1.0f);
    } else if (k == 0u) {                          // Square
        y = x < o.half ? 1.0f : -1.0f;
    } else if (k == 2u) {                          // Triangle
        const float a = __fmaf_rn(o.ts1, x, 1.0f);
        const float b = __fmaf_rn(o.ts2, __fsub_rn(x, o.half), -1.0f);
        y = x < o.half ? a : b;
    } else {                                       // Sine: try3/lookup.rs:46-85 on SIN_TABLE
        const float tv = __fdiv_rn(__fmul_rn(x, 1024.0f), o.P);
        const uint32_t i1 = __float2uint_rz(tv);   // `as u32`: truncating, saturating
        const uint32_t i2 = (i1 + 1u) & 1023u;
        const float s1 = i1 < 1024u ? sintab[i1] : 0.0f;   // gather_or_default
        const float s2 = sintab[i2];
        y = __fmaf_rn(__fsub_rn(s2, s1), __fsub_rn(tv, __uint2float_rn(i1)), s1);
    }
    const float t = __fadd_rn(ph, o.d);
    if (LITERAL) ph = fmodf(t, 1.0f);
    else ph = wrap_unit(t);
    return y;
}

// try3/hashnoise.rs:33-68.  value / 65535 is replaced by fma(v, 0x1.0001p-16, 2^-45): v * 0x1.0001p-16 is exact in
// the fma and lies below the true quotient by less than 2^-32, with no rounding boundary in between except
// when it sits on one itself (a tie), which the tiny addend resolves upwards as the true quotient would be:
// equal to the IEEE quotient for all 65,536 possible values (tests/test_oracle_kats.py).
// (q * 2) - 1 is one fma because q * 2 is exact.
constexpr float kNoiseHi = 0x1.0001p-16f, kNoiseEps = 0x1p-45f;
__device__ __forceinline__ uint32_t noise_hash(uint32_t rot, uint32_t n) { return (rot ^ n) * 0x9e3779b9u; }
__device__ __forceinline__ float noise_fast(uint32_t rot, uint32_t n) {
    const float v = __uint2float_rn(noise_hash(rot, n) & 0xffffu);
    const float q = __fmaf_rn(v, kNoiseHi, kNoiseEps);
    return __fmaf_rn(q, 2.0f, -1.0f);
}

__device__ __forceinline__ float noise_literal(uint32_t rot, uint32_t n) {
    const uint32_t off = __float2uint_rz(__uint2float_rn(n));   // u32 -> f32 -> u32 (process.rs:347-348)
    const uint32_t h = (rot ^ off) * 0x9e3779b9u;
    const float v = __uint2float_rn(h & 0xffffu);
    const float q = __fdiv_rn(v, 65535.0f);
    return __fsub_rn(__fmul_rn(q, 2.0f), 1.0f);
}

template <int FILTER>
__device__ __forceinline__ float filt_step(float u, const FiltC& c, FiltS& s) {
    if (FILTER == 0) {
        // try3/filters.rs:23-33: a0.mul_add(input, -b1 * last), b1 = -k
        const float y = __fmaf_rn(c.c1, u, __fmul_rn(c.c0, s.y1));
        s.y1 = y;
        return y;
    } else if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP || FILTER == FILT_BIQUAD_BP) {
        // try3/dsp_filters.rs:116-128: 2*(alpha*(x + 2*x1 + x2) + gamma*y1 - beta*y2); x + 2*x1 is one fma
        // because 2*x1 is exact.  :166-176 (high-pass) has x - 2*x1 + x2, :214-224 (band-pass) x - x2.
        float sx;
        if (FILTER == FILT_BIQUAD_LP) sx = __fadd_rn(__fmaf_rn(2.0f, s.x1, u), s.x2);
        else if (FILTER == FILT_BIQUAD_HP) sx = __fadd_rn(__fmaf_rn(-2.0f, s.x1, u), s.x2);
        else sx = __fsub_rn(u, s.x2);
        float t = __fmul_rn(c.c0, sx);
        t = __fadd_rn(t, __fmul_rn(c.c2, s.y1));
        t = __fsub_rn(t, __fmul_rn(c.c1, s.y2));
        s.x2 = s.x1; s.x1 = u; s.y2 = s.y1; s.y1 = t;
        return t;
    } else {
        // try3/dsp_filters.rs:37-41 / :71-75: alpha * (x +- x1) + gamma * y1 (no mul_add in the source)
        const float xs = FILTER == FILT_FIRST_LP ? __fadd_rn(u, s.x1) : __fsub_rn(u, s.x1);
        const float t = __fadd_rn(__fmul_rn(c.c0, xs), __fmul_rn(c.c2, s.y1));
        s.x1 = u; s.y1 = t;
        return t;
    }
}

// Two frames of the filter, u2 = inputs of frames (i, i + 1), with per-frame coefficients ca / cb (the same
// object twice on the fast path).  Same operations as filt_step twice; the feed-forward product c0 * sx of the
// second-order filters is computed for both frames in one packed multiply (it feeds scalar adds only: no
// contraction, see the hazard note below).
template <int FILTER>
__device__ __forceinline__ float2 filt_step2(float2 u2, const FiltC& ca, const FiltC& cb, FiltS& s) {
    if (FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP || FILTER == FILT_BIQUAD_BP) {
        float sxa, sxb;
        if (FILTER == FILT_BIQUAD_LP) {
            sxa = __fadd_rn(__fmaf_rn(2.0f, s.x1, u2.x), s.x2);
            sxb = __fadd_rn(__fmaf_rn(2.0f, u2.x, u2.y), s.x1);
        } else if (FILTER == FILT_BIQUAD_HP) {
            sxa = __fadd_rn(__fmaf_rn(-2.0f, s.x1, u2.x), s.x2);
            sxb = __fadd_rn(__fmaf_rn(-2.0f, u2.x, u2.y), s.x1);
        } else {
            sxa = __fsub_rn(u2.x, s.x2);
            sxb = __fsub_rn(u2.y, s.x1);
        }
        const float2 p = s2c::vmul(make_float2(ca.c0, cb.c0), make_float2(sxa, sxb));
        float ta = __fadd_rn(p.x, __fmul_rn(ca.c2, s.y1));
        ta = __fsub_rn(ta, __fmul_rn(ca.c1, s.y2));
        float tb = __fadd_rn(p.y, __fmul_rn(cb.c2, ta));
        tb = __fsub_rn(tb, __fmul_rn(cb.c1, s.y1));
        s.x2 = u2.x; s.x1 = u2.y; s.y2 = ta; s.y1 = tb;
        return make_float2(ta, tb);
    } else {
        const float ya = filt_step<FILTER>(u2.x, ca, s);
        const float yb = filt_step<FILTER>(u2.y, cb, s);
        return make_float2(ya, yb);
    }
}

// ------------------------------------------------------------------------------------------
// Packed arithmetic: Blackwell's FADD2 / FMUL2 / FFMA2 retire two IEEE-754 round-to-nearest results per issue
// slot — the render loop is issue-bound, not FLOP-bound (profiles/r1_notes.md).  Each element is rounded exactly
// like the scalar instruction, so parity is unchanged.
//
// CONTRACTION HAZARD (ptxas 12.9, sm_100a): a packed multiply whose result feeds a packed add is fused
// into FFMA2 — with the __fmul2_rn/__fadd2_rn builtins AND with explicit `mul.rn.f32x2` / `add.rn.f32x2`
// PTX, -fmad=false notwithstanding (tools/ubench/fuse_check.cu; scalar __fmul_rn + __fadd_rn is not
// fused).  That moves results by an ulp and can flip a square wave's sign.  Rule used in this file: the
// result of pmul2 never feeds padd2; where the reference adds to a rounded product, the add is either scalar
// __fadd_rn per element or s2c::vaddp (an fma with a multiplicand of 1 that ptxas cannot see through).
__device__ __forceinline__ float2 padd2(float2 a, float2 b) { return s2c::vadd(a, b); }
__device__ __forceinline__ float2 pmul2(float2 a, float2 b) { return s2c::vmul(a, b); }
__device__ __forceinline__ float2 pfma2(float2 a, float2 b, float2 c) { return s2c::vfma(a, b, c); }
__device__ __forceinline__ float2 splat2(float x) { return make_float2(x, x); }

// Per-lane constants and state of the fast paths (registers).
struct FastV {
    // oscillator (derived from the period; negations are stored so the loop only adds)
    float P, d, slope, nhalf, ts1, ts2;
    // patch
    float gain, namt;
    // filter of a resting cutoff (fl_bits unused)
    FiltC fc;
    // amp envelope segment of the lane's current frame: g = es * (x + nex0) + ey0 for frame offsets [.., seg_end)
    float es, nex0, ey0;
    uint32_t seg_end;
    // carried state
    float ph;
    FiltS fs;
};

__device__ __forceinline__ void set_osc(FastV& F, const OscC& o) {
    F.P = o.P; F.d = o.d; F.slope = o.slope; F.nhalf = -o.half; F.ts1 = o.ts1; F.ts2 = o.ts2;
}
__device__ __forceinline__ OscC osc_of(const FastV& F) {
    OscC o;
    o.P = F.P; o.d = F.d; o.slope = F.slope; o.half = -F.nhalf; o.ts1 = F.ts1; o.ts2 = F.ts2; o.fo_bits = 0;
    return o;
}

// es * (x + nex0) + ey0 for frames (x.x, x.y): an envelope segment's line (SegEnv), the add through an fma by one
// (see the hazard note)
__device__ __forceinline__ float2 seg_line2(float es, float nex0, float ey0, float2 x, float one) {
    return s2c::vaddp(pmul2(splat2(es), padd2(x, splat2(nex0))), splat2(ey0), one);
}

// How a chunk evaluates the amp envelope.
enum { G_CONST = 0,      // every frame of the chunk lies in a segment of slope 0 (sustain, end): g = ey0
       G_LINE = 1,       // every frame lies in the lane's current segment: one line, two frames per instruction
       G_ANY = 2 };      // a stage boundary falls inside the chunk for some lane: per pair, the full stage chain at boundaries

// The amp envelope of frames (x, x + 1) where a stage boundary falls on or between them: the full stage chain for
// both, then the segment of the frame after them.  Out of line: it runs a handful of times per voice per render.
struct AmpEdge { float2 g; SegEnv sg; };
static __device__ __noinline__ AmpEdge amp_at_boundary(const EnvQ* __restrict__ amp, float xa, float xb, uint32_t n_next) {
    const EnvQ A = *amp;
    AmpEdge e;
    e.g = make_float2(env_x16(A, xa), env_x16(A, xb));
    e.sg = seg_env(A, n_next);
    return e;
}

// Waveform of frames (i, i + 1) from their phases, period constant (the `% period` is a no-op, see osc_step).
template <int KIND>
__device__ __forceinline__ float2 wave2(const FastV& F, float2 ph2, float hbig, uint32_t kind, const float* sintab) {
    const float2 x2 = pmul2(splat2(F.P), ph2);                 // period.mul_add(phase, 0)
    float2 osc2;
    if (KIND == 1) {
        osc2 = pfma2(splat2(F.slope), x2, splat2(1.0f));
    } else if (KIND == 0) {
        // x < P/2 ? +1 : -1 without a compare or bit surgery: s = sat(2^60 * (P/2 - x)) is exactly 1 when
        // x < P/2 and exactly 0 otherwise (the fma is exact in sign; two distinct binary32 values of this
        // magnitude differ by >= 2^-24, so the product is >= 2^36 before the clamp; equality gives +0; a
        // NaN clamps to 0, i.e. -1, as `NaN < h` is false), and 2 s - 1 is exact.
        const float2 sq = make_float2(__saturatef(__fmaf_rn(x2.x, -0x1p60f, hbig)),
                                      __saturatef(__fmaf_rn(x2.y, -0x1p60f, hbig)));
        osc2 = pfma2(sq, splat2(2.0f), splat2(-1.0f));
    } else if (KIND == 2) {
        const float2 dl = make_float2(__fadd_rn(x2.x, F.nhalf), __fadd_rn(x2.y, F.nhalf));
        const float2 a = pfma2(splat2(F.ts1), x2, splat2(1.0f));
        const float2 b = pfma2(splat2(F.ts2), dl, splat2(-1.0f));
        osc2.x = dl.x < 0.0f ? a.x : b.x;
        osc2.y = dl.y < 0.0f ? a.y : b.y;
    } else {
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const uint32_t k = KIND == 3 ? 3u : kind;
            const float xe = e ? x2.y : x2.x, he = -F.nhalf;
            float y;
            if (k == 1u) y = __fmaf_rn(F.slope, xe, 1.0f);
            else if (k == 0u) y = xe < he ? 1.0f : -1.0f;
            else if (k == 2u) {
                const float a = __fmaf_rn(F.ts1, xe, 1.0f);
                const float b = __fmaf_rn(F.ts2, __fsub_rn(xe, he), -1.0f);
                y = xe < he ? a : b;
            } else {                                       // try3/lookup.rs:46-85 on SIN_TABLE
                const float tv = __fdiv_rn(__fmul_rn(xe, 1024.0f), F.P);
                const uint32_t i1 = __float2uint_rz(tv);
                const uint32_t i2 = (i1 + 1u) & 1023u;
                const float s1 = i1 < 1024u ? sintab[i1] : 0.0f;
                const float s2 = sintab[i2];
                y = __fmaf_rn(__fsub_rn(s2, s1), __fsub_rn(tv, __uint2float_rn(i1)), s1);
            }
            if (e) osc2.y = y; else osc2.x = y;
        }
    }
    return osc2;
}

// Noise of two frames from their hash words, and the filter input u = (osc + gain) + (noise + amount)
// (process.rs:341-358: gain and amount are ADDED on the x16 path; nz + 0.0 == nz bit-for-bit, so NAMT0 drops it)
template <bool NAMT0>
__device__ __forceinline__ float2 input2(const FastV& F, float2 osc2, uint32_t ha, uint32_t hb) {
    const float2 v2 = make_float2(__uint2float_rn(ha & 0xffffu), __uint2float_rn(hb & 0xffffu));
    const float2 q2 = pfma2(v2, splat2(kNoiseHi), splat2(kNoiseEps));
    const float2 nz2 = pfma2(q2, splat2(2.0f), splat2(-1.0f));
    return padd2(padd2(osc2, splat2(F.gain)), NAMT0 ? nz2 : padd2(nz2, splat2(F.namt)));
}

// The filter input of one frame, u = (osc + gain) + (noise + amount), as input2
__device__ __forceinline__ float input1(const FastV& F, float osc, uint32_t rot, uint32_t n) {
    return __fadd_rn(__fadd_rn(osc, F.gain), __fadd_rn(noise_fast(rot, n), F.namt));
}

// One frame of one voice, x16 semantics in the fast forms (osc_step without the `%`, noise_fast), filter coefficients
// c: the phase step, waveform, filter input and filter step.  Returns the filter's output.
template <int FILTER, int KIND>
__device__ __forceinline__ float voice_frame(FastV& F, const FiltC& c, uint32_t kind, uint32_t rot, uint32_t n,
                                             const float* sintab) {
    const float osc = osc_step<KIND, false>(kind, osc_of(F), F.ph, sintab);
    return filt_step<FILTER>(input1(F, osc, rot, n), c, F.fs);
}

// Frames (i, i + 1) of one voice in the time-packed loops, filter coefficients ca / cb and noise hash words ha / hb of
// the two frames.  The two recurrences (phase, filter) stay scalar — a packed op has twice the latency — while
// everything that is feed-forward (waveform, noise map, gain / noise combine, the filter's input product, output gain)
// is computed for both frames in one packed instruction.  Element-wise rounding is identical to the scalar form.
// gain() gives the amp envelope of the two frames, evaluated after the filter step.  hbig = (P / 2) * 2^60 (wave2).
template <int FILTER, int KIND, bool NAMT0, int TRACE, class Gain>
__device__ __forceinline__ float2 voice_pair(FastV& F, const FiltC& ca, const FiltC& cb, uint32_t ha, uint32_t hb,
                                             float hbig, uint32_t kind, const float* sintab, Gain&& gain) {
    // phase recurrence, two frames (try3/oscillators.rs:377-381; see osc_step)
    const float pa = F.ph;
    const float pb = wrap_unit(__fadd_rn(pa, F.d));
    F.ph = wrap_unit(__fadd_rn(pb, F.d));
    const float2 ph2 = make_float2(pa, pb);
    const float2 osc2 = wave2<KIND>(F, ph2, hbig, kind, sintab);
    const float2 y2 = filt_step2<FILTER>(input2<NAMT0>(F, osc2, ha, hb), ca, cb, F.fs);
    // envelope (old/simdtest.rs:270-330) and output gain (process.rs:373-378)
    const float2 g2 = gain();
    return TRACE == TRACE_PHASE ? ph2 : pmul2(y2, g2);
}

// Time-packed fast chunk: 32 frames of one voice per lane with period, cutoff and (G_CONST / G_LINE) amp-envelope
// segment constant, two frames per step (voice_pair).
// FASTHASH: the noise amount is +0.0 and the voice's frame offset and rotated seed are multiples of 8 (seeds below
// 2^27 rotate to multiples of 32), so (seed' ^ (offset + i)) == (seed' ^ offset) + i and the hash of frame i is one
// add with an immediate.
template <int FILTER, int KIND, int GMODE, bool FASTHASH, int TRACE>
__device__ __forceinline__ void chunk_fast_tp(FastV& F, const EnvQ* __restrict__ amp, float one, uint32_t kind, uint32_t rot,
                                              uint32_t n0, float* __restrict__ row, const float* sintab) {
    const float hbig = __fmul_rn(-F.nhalf, 0x1p60f);               // (P / 2) * 2^60, exact
    uint32_t n = n0;
    float2 xf2 = make_float2(__uint2float_rn(n0), __uint2float_rn(n0 + 1u));       // exact: n0 + 32 <= 2^24
    SegEnv sg = {0.0f, 0.0f, 0.0f, 0u, 0u, 0};
    if (GMODE == G_ANY) sg = seg_env(*amp, n0);
    // 8 frames per trip: long enough to overlap neighbouring frames, short enough for the instruction cache
#pragma unroll 1
    for (int jt = 0; jt < kChunk / S2_TRIP; jt++) {
    // FASTHASH: nb ^ i == nb + i for i < 8, so the hash of frame i is nb * C + i * C: one multiply per trip and
    // one add with an immediate per frame
    const uint32_t nbc = noise_hash(rot, n);
#pragma unroll
    for (int jj = 0; jj < S2_TRIP / 4; jj++) {
        const int j = (S2_TRIP / 4) * jt + jj;
        float o4[4];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const uint32_t fi = 4u * jj + 2u * h;                 // frame index inside the trip (compile-time)
            const uint32_t ha = FASTHASH ? nbc + fi * 0x9e3779b9u : noise_hash(rot, n + fi);
            const uint32_t hb = FASTHASH ? nbc + (fi + 1u) * 0x9e3779b9u : noise_hash(rot, n + fi + 1u);
            const float2 out2 = voice_pair<FILTER, KIND, FASTHASH, TRACE>(F, F.fc, F.fc, ha, hb, hbig, kind, sintab, [&] {
                if (GMODE == G_CONST) return splat2(F.ey0);
                float2 g2;
                if (GMODE == G_LINE) {
                    g2 = seg_line2(F.es, F.nex0, F.ey0, xf2, one);
                } else if (n + fi + 2u <= sg.nend) {
                    // both frames inside the current segment: its line, bit-exact (see SegEnv)
                    g2 = make_float2(seg_eval(sg, xf2.x), seg_eval(sg, xf2.y));
                } else {
                    const AmpEdge e = amp_at_boundary(amp, xf2.x, xf2.y, n + fi + 2u);
                    g2 = e.g;
                    sg = e.sg;
                }
                xf2 = padd2(xf2, splat2(2.0f));
                return g2;
            });
            o4[2 * h] = out2.x;
            o4[2 * h + 1] = out2.y;
        }
        *reinterpret_cast<float4*>(row + 4 * j) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    }
    n += (uint32_t)S2_TRIP;
    }
}

// Per-lane inputs of a moving-cutoff chunk (registers, valid for one chunk).
struct MovV {
    CutP cp;
    float mes, mnex0, mey0;      // the mod envelope's segment line (the whole chunk lies inside it)
    bool moving;                 // false: this lane's cutoff rests (F.fc) while others of the warp move
};

// Moving-cutoff chunk, packed: the period is constant but the mod envelope is in a ramp, so the cutoff — and with
// it the filter coefficients — changes every frame (process.rs:148-152, 363-371; the first 200 ms of every note of
// the default patch, synth.rs:141-150).  Preconditions (the classifier checks them for every lane): the chunk lies
// inside the lane's current amp-envelope segment (F.es .., as G_LINE); for every MOVING lane it starts at a multiple
// of 32 frames, lies inside one segment of the mod envelope, and (second-order filters) its window W is valid.
// Every frame's coefficients come from the reference's own chain, two frames per instruction (s2_cutoff.h): 2^x
// around the window's centre, the angle, sin / cos by angle addition, the coefficient algebra.  The one-pole
// evaluates k = e^-theta every frame.  Lanes whose cutoff rests run the same code and select their constants.
// ONE variant per oscillator kind and 4 frames per trip, on purpose: a moving-cutoff step walks through the
// classifier, the window's binary64 code, this loop and the write-back once per chunk, and with 8-frame trips in
// four variants that path outgrew the 32 KB instruction cache of an SM — 41 % of the stall samples of such a launch
// were instruction fetch (profiles/r2_notes.md).
// SHARED: the warp's voices share one cutoff trajectory and the chunk's 32 coefficient sets are in `ctab`
// ([c0 | c1 | c2][32], modcut_coefficients): the loop reads them, two frames per load, instead of evaluating them.
template <int FILTER, int KIND, int TRACE, bool SHARED = false>
__device__ __forceinline__ void chunk_modcut_pk(FastV& F, const MovV& mv, const s2c::Window& W,
                                                float one, uint32_t kind, uint32_t rot, uint32_t n0,
                                                float* __restrict__ row, const float* sintab,
                                                const float* __restrict__ ctab = nullptr) {
    static_assert(SHARED || FILTER == FILT_ONE_POLE || FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP, "packed moving-cutoff filters");
    const float hbig = __fmul_rn(-F.nhalf, 0x1p60f);
    uint32_t n = n0;
    float2 xf2 = make_float2(__uint2float_rn(n0), __uint2float_rn(n0 + 1u));
#pragma unroll 1
    for (int j = 0; j < kChunk / 4; j++) {
        float o4[4];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            // the mod envelope's line at the two frame offsets
            const float2 m2 = seg_line2(mv.mes, mv.mnex0, mv.mey0, xf2, one);
            float2 c0, c1, c2;
            if (SHARED) {
                c0 = *reinterpret_cast<const float2*>(ctab + 4 * j + 2 * h);
                c1 = *reinterpret_cast<const float2*>(ctab + 32 + 4 * j + 2 * h);
                c2 = *reinterpret_cast<const float2*>(ctab + 64 + 4 * j + 2 * h);
            } else if (FILTER == FILT_ONE_POLE) {
                c0 = s2c::exp_neg_fast<float2>(s2c::theta_at<float2>(m2, mv.cp.amt, mv.cp.theta0));
                c1 = pfma2(c0, splat2(-one), splat2(1.0f));               // 1 - k, one rounding (exact product)
                c2 = splat2(0.0f);
            } else {
                float2 s2, co2;
                window_frame_sincos<float2>(W, mv.cp, one, m2, &s2, &co2);
                s2c::biquad_lp_hp<FILTER == FILT_BIQUAD_HP, float2>(s2, co2, mv.cp.hd, one, &c0, &c1, &c2);
            }
            if (!mv.moving) { c0 = splat2(F.fc.c0); c1 = splat2(F.fc.c1); c2 = splat2(F.fc.c2); }
            const FiltC ca = {c0.x, c1.x, c2.x, 0u}, cb = {c0.y, c1.y, c2.y, 0u};
            const float2 out2 = voice_pair<FILTER, KIND, false, TRACE>(F, ca, cb, noise_hash(rot, n), noise_hash(rot, n + 1u),
                                                                       hbig, kind, sintab,
                                                                       [&] { return seg_line2(F.es, F.nex0, F.ey0, xf2, one); });
            o4[2 * h] = out2.x;
            o4[2 * h + 1] = out2.y;
            n += 2u;
            xf2 = padd2(xf2, splat2(2.0f));
        }
        *reinterpret_cast<float4*>(row + 4 * j) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    }
}

// The same chunk when no aligned lane pair (2i, 2i + 1) holds two moving lanes (s2_bank_create lays the slots out that
// way where it can): the resting lane of a pair computes half of its partner's coefficients instead of idling.  Per
// trip of 4 frames every lane evaluates ONE pair of frames of its ASSIGNED voice — its own if it moves (frames 4j,
// 4j + 1), its partner's if it helps (frames 4j + 2, 4j + 3) — up to (q, cos), the pair swaps them by a shuffle, and
// every lane finishes both pairs' coefficient algebra and runs its own voice.  The same functions on the same
// operands as chunk_modcut_pk, hence the same bits; a third fewer arithmetic instructions per frame.
template <int FILTER, int KIND, int TRACE>
__device__ __forceinline__ void chunk_modcut_pr(FastV& F, const MovV& mv, const s2c::Window& W,
                                                float one, uint32_t kind, uint32_t rot, uint32_t n0,
                                                float* __restrict__ row, const float* sintab) {
    static_assert(FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP, "paired moving-cutoff filters");
    constexpr uint32_t kAll = 0xffffffffu;
    const bool partner_moves = __shfl_xor_sync(kAll, (int)mv.moving, 1) != 0;      // (every lane runs every shuffle)
    const bool helper = !mv.moving && partner_moves;
    auto assigned = [&](float v) { const float t = __shfl_xor_sync(kAll, v, 1); return helper ? t : v; };
    // the assigned voice: cutoff constants, window, mod-envelope line, frame offset of the first assigned pair
    CutP cp = mv.cp;
    cp.lpf = assigned(mv.cp.lpf); cp.amt = assigned(mv.cp.amt); cp.hd = assigned(mv.cp.hd);
    s2c::Window Wa = W;
    Wa.xc = assigned(W.xc); Wa.Eh = assigned(W.Eh); Wa.Er = assigned(W.Er); Wa.thc = assigned(W.thc);
    Wa.Ah = assigned(W.Ah); Wa.Al = assigned(W.Al); Wa.Bh = assigned(W.Bh); Wa.Bl = assigned(W.Bl);
    const float mes = assigned(mv.mes), mnex0 = assigned(mv.mnex0), mey0 = assigned(mv.mey0);
    const float xa = __fadd_rn(assigned(__uint2float_rn(n0)), helper ? 2.0f : 0.0f);
    float2 xa2 = make_float2(xa, __fadd_rn(xa, 1.0f));

    const float hbig = __fmul_rn(-F.nhalf, 0x1p60f);
    uint32_t n = n0;
    float2 xf2 = make_float2(__uint2float_rn(n0), __uint2float_rn(n0 + 1u));
#pragma unroll 1
    for (int j = 0; j < kChunk / 4; j++) {
        const float2 m2 = seg_line2(mes, mnex0, mey0, xa2, one);
        float2 s2, co2;
        window_frame_sincos<float2>(Wa, cp, one, m2, &s2, &co2);
        const float2 q2 = s2c::quotient_of<float2>(s2, cp.hd, one);
        xa2 = padd2(xa2, splat2(4.0f));
        // the partner's pair: a moving lane receives its frames 4j + 2, 4j + 3
        const float2 qo = make_float2(__shfl_xor_sync(kAll, q2.x, 1), __shfl_xor_sync(kAll, q2.y, 1));
        const float2 coo = make_float2(__shfl_xor_sync(kAll, co2.x, 1), __shfl_xor_sync(kAll, co2.y, 1));
        float o4[4];
#pragma unroll
        for (int h = 0; h < 2; h++) {
            float2 c0, c1, c2;
            s2c::biquad_from_q_cos<FILTER == FILT_BIQUAD_HP, float2>(h ? qo : q2, h ? coo : co2, one, &c0, &c1, &c2);
            if (!mv.moving) { c0 = splat2(F.fc.c0); c1 = splat2(F.fc.c1); c2 = splat2(F.fc.c2); }
            const FiltC ca = {c0.x, c1.x, c2.x, 0u}, cb = {c0.y, c1.y, c2.y, 0u};
            const float2 out2 = voice_pair<FILTER, KIND, false, TRACE>(F, ca, cb, noise_hash(rot, n), noise_hash(rot, n + 1u),
                                                                       hbig, kind, sintab,
                                                                       [&] { return seg_line2(F.es, F.nex0, F.ey0, xf2, one); });
            o4[2 * h] = out2.x;
            o4[2 * h + 1] = out2.y;
            n += 2u;
            xf2 = padd2(xf2, splat2(2.0f));
        }
        *reinterpret_cast<float4*>(row + 4 * j) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    }
}

// Moving-cutoff chunk, one frame at a time: any alignment, any filter, windows made on demand (valid or not).
// The chunk lies inside one segment `sm` of the mod envelope.  The same per-frame functions as the packed form,
// hence the same bits.
// SHARED: every voice of the warp has the same cutoff trajectory (same cutoff, damping, modulation amount, mod
// envelope and frame offset — a detune / pitch sweep of one patch, BASELINE config 5), so the 32 frames'
// coefficients were computed once, one frame per lane, into `ctab` ([c0 | c1 | c2][32], see modcut_coefficients).
template <int FILTER, int KIND, int TRACE, bool SHARED>
__device__ __forceinline__ void chunk_modcut_sc(FastV& F, const EnvQ* __restrict__ amp, const MovV& mv, const SegEnv& sm,
                                                float one, uint32_t kind, uint32_t rot, uint32_t n0,
                                                float* __restrict__ row, const float* sintab, const float* __restrict__ ctab) {
    SegEnv sa = seg_env(*amp, n0);
    FiltC fc = F.fc;
    s2c::Window W;
    window_none(W);
    uint32_t n = n0;
    float xf = __uint2float_rn(n0);                               // exact: n0 + 32 <= 2^24
#pragma unroll 1
    for (int i = 0; i < kChunk; i++) {
        const float g = seg_walk(sa, *amp, n, xf);
        if (SHARED) { fc.c0 = ctab[i]; fc.c1 = ctab[32 + i]; fc.c2 = ctab[64 + i]; }
        else if (mv.moving) moving_coefs<FILTER>(fc, W, sm, mv.cp, one, n, seg_eval(sm, xf));
        const float ph0 = F.ph;
        const float y = voice_frame<FILTER, KIND>(F, fc, kind, rot, n, sintab);
        row[i] = TRACE == TRACE_PHASE ? ph0 : __fmul_rn(y, g);
        n += 1u;
        xf = __fadd_rn(xf, 1.0f);
    }
}

// One frame per lane: the filter coefficients of frames n0 .. n0 + 31 of a cutoff trajectory shared by the warp.
template <int FILTER>
__device__ __forceinline__ void modcut_coefficients(const SegEnv& sm, const CutP& cp, float one, uint32_t n0, int lane,
                                                    float* __restrict__ ctab) {
    const uint32_t n = n0 + (uint32_t)lane;
    s2c::Window W;
    window_none(W);
    FiltC c;
    moving_coefs<FILTER>(c, W, sm, cp, one, n, seg_eval(sm, __uint2float_rn(n)));
    ctab[lane] = c.c0; ctab[32 + lane] = c.c1; ctab[64 + lane] = c.c2;
}

// Moving-cutoff state of the general per-frame path (one voice, any frame order inside a chunk)
struct MovG {
    CutP cp;
    SegEnv sm;           // the mod-envelope segment of the last moving frame (nbeg > nend: none yet)
    s2c::Window W;
};
__device__ __forceinline__ void movg_init(MovG& g, float lpf, float amt_lpf, float damp, float sr) {
    g.cp = make_cutp(lpf, amt_lpf, damp, sr);
    g.sm.nbeg = 1u; g.sm.nend = 0u; g.sm.es = g.sm.nex0 = g.sm.ey0 = 0.0f; g.sm.stage = 4;
    window_none(g.W);
}

// Filter coefficients of x16 frame n (m = its mod-envelope value): the moving evaluation while the mod envelope ramps
// and the cutoff follows it, the resting one (memoised by the cutoff's bits) otherwise.  Below 2^24 the frame offset
// is exact in f32 and the segment arithmetic holds; beyond, the envelope rests anyway.
template <int FILTER>
__device__ __forceinline__ void x16_coefs(FiltC& c, MovG& mg, const EnvP& M, float lpf, float amt_lpf, float damp,
                                          float sr, float one, uint32_t n, float m) {
    bool moving = false;
    if (amt_lpf != 0.0f && n < (1u << 24)) {
        if (n < mg.sm.nbeg || n >= mg.sm.nend) mg.sm = seg_env(M, n);
        moving = stage_moves(mg.sm.stage);
    }
    if (moving) {
        moving_coefs<FILTER>(c, mg.W, mg.sm, mg.cp, one, n, m);
    } else {
        const float fl = modulate_freq(lpf, m, amt_lpf);
        if (__float_as_uint(fl) != c.fl_bits) make_filt<FILTER>(c, fl, damp, sr);
    }
}

// General frame: the normative per-sample semantics (SURVEY.md section 8a), x16 or scalar-tail flavour.
template <int FILTER, int TRACE>
__device__ __forceinline__ float general_frame(const Lane& L, float sr, float one, uint32_t n, bool scalar_sem, OscC& o,
                                               FiltC& c, MovG& mg, float& ph, FiltS& fs, const float* sintab) {
    const float x = __uint2float_rn(n);           // offset as f32
    float g, m;
    if (!scalar_sem) { g = env_x16(L.amp, x); m = env_x16(L.mod, x); }
    else { g = env_scalar(L.amp, x); m = env_scalar(L.mod, x); }
    const float fo = modulate_freq(L.pitch, m, L.amt_osc);
    if (__float_as_uint(fo) != o.fo_bits) make_osc(o, fo, sr);
    if (!scalar_sem) {
        x16_coefs<FILTER>(c, mg, L.mod, L.lpf, L.amt_lpf, L.damp, sr, one, n, m);
    } else {
        const float fl = modulate_freq(L.lpf, m, L.amt_lpf);
        if (__float_as_uint(fl) != c.fl_bits) make_filt<FILTER>(c, fl, L.damp, sr);
    }
    const float ph0 = ph;
    const float osc = osc_step<-1, true>(L.kind, o, ph, sintab);
    const float nz = noise_literal(L.rot, n);
    float u;
    if (!scalar_sem) u = __fadd_rn(__fadd_rn(osc, L.gain), __fadd_rn(nz, L.namt));
    else u = __fadd_rn(__fmul_rn(osc, L.gain), __fmul_rn(nz, L.namt));   // process.rs:287-294
    const float y = filt_step<FILTER>(u, c, fs);
    return TRACE == TRACE_PHASE ? ph0 : __fmul_rn(y, g);
}

// ------------------------------------------------------------------------------------------

// Per-voice state that only the classifier, the general path and the epilogue touch.  It lives in
// shared memory ("coefficient and state tiles"), not in registers: the fast loops then own the whole
// register budget that keeps all 13.8 warps per SM resident.  An odd word count keeps the 32
// lanes of a warp on distinct banks.
struct Cold {
    EnvQ amp, mod;         // the envelopes as the x16 path evaluates them (the scalar tail re-derives the full form)
    float pitch, lpf, damp, amt_osc, amt_lpf;
    float theta0;          // (2 pi cutoff) / sr
    OscC oc;
    FiltC fc;
    SegEnv msg;            // the mod-envelope ramp the voice's moving cutoff is in (flags bit 2)
    uint32_t release;      // release offset in force for this launch (the parameter row or a staged note-off table)
    uint32_t n_safe;       // the resting constants (period, cutoff) are valid for frame offsets [.., n_safe)
    uint32_t vi;           // slot index (state/params column)
    uint32_t out_row;      // caller-visible voice index, 0xffffffff = no such voice
    uint32_t flags;        // bit 0 active, bit 1 mod envelope matters, bit 2 the cutoff is moving (see msg)
};
constexpr int kColdWords = (sizeof(Cold) / 4) | 1;
constexpr int kRowPtrWords = 2;    // one 64-bit output-row base per tile row (0 = the row has no output)
constexpr int kCoefWords = 96;     // shared moving-cutoff coefficients of one chunk: [c0 | c1 | c2][32]

__host__ __device__ constexpr size_t warp_smem_floats() {
    return 32 * kTileStride + 32 * kColdWords + 32 * kRowPtrWords + kCoefWords;      // 14.8 KB: 14 one-warp blocks per SM
}

}  // namespace s2
