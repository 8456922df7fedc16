// check_cutoff.cpp — CPU check of synth2_b200/csrc/s2_cutoff.h (the scalar forms of what the kernels compile).
//   g++ -O2 -std=c++17 -ffp-contract=off -march=x86-64-v3 -o check_cutoff tools/check_cutoff.cpp && ./check_cutoff [quick]
// 1. div_in_range against the IEEE quotient over the operand range of the second-order filters, with the reciprocal
//    estimate off by up to +-2 ulp (the special-function unit's error is not modelled more finely than that): how
//    often it is not the correctly rounded value, and by how much;
// 2. exp_neg_fast against exp(-theta) in binary64; at theta = +inf (an overflowing cutoff) it is 0, and its clamp
//    against the unclamped form for every binary32 theta (every 61st in quick mode);
// 3. windowed sin / cos against the once-rounded binary64 values: mismatch rates and worst absolute error;
// 4. theta_of (division by the sample rate as reciprocal + residual step) against the IEEE quotient, for EVERY binary32
//    numerator the path can produce, at the usual rates;
// 5. sweep_exact (2^x around a window's centre) against 2^x rounded once;
// 6. a whole decay sweep of the resonant low-pass at its worst corner (100-200 Hz, damping 0.2): coefficients from
//    windows vs the full per-frame evaluation (the reference's chain with binary64 transcendentals rounded once),
//    and the filter outputs they produce.
// Exits non-zero if 1 is off by more than an ulp or wrong in more than 1e-4 of the cases, if 2 exceeds 4 ulp, gives
// anything but 0 at +inf or changes a bit of the unclamped form below the clamp, if 3 adds
// more than 4e-9 to a correct rounding (or misses the rounded-once value in more than 2 % of slow-sweep frames), if 4
// differs anywhere, if 5 differs in more than 1 % of arguments or by more than an ulp, or if 6 changes a coefficient
// in more than 2 % of the frames.
#include "../synth2_b200/csrc/s2_cutoff.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>

using namespace s2c;

static uint32_t bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static float fbits(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

static void make_window(Window& W, float thc) {
    W.k = 0; W.valid = 1; W.thc = thc;
    double s, c; s2_sincos_d((double)thc, &s, &c);
    split_hi_lo(s, &W.Ah, &W.Al); split_hi_lo(c, &W.Bh, &W.Bl);
}

int main(int argc, char** argv) {
    const bool quick = argc > 1 && !strcmp(argv[1], "quick");
    int fail = 0;

    // ---- 1. division
    {
        std::mt19937_64 rng(12345);
        long n = 0, bad = 0, worse = 0;
        const long N = quick ? 4000000 : 40000000;
        for (long i = 0; i < N; i++) {
            const float h = (float)((rng() >> 11) * (1.0 / 9007199254740992.0)) * 8.0f;      // hd * sin in [0, 8)
            const float num = 1.0f - h, den = 1.0f + h, nden = -1.0f - h;
            const float want = num / den;
            const float r0 = 1.0f / den;
            for (int p = -2; p <= 2; p++) {
                const float r = fbits(bits(r0) + (uint32_t)p);
                const float got = div_in_range_from<float>(num, nden, r);
                n++;
                if (bits(got) != bits(want)) {
                    bad++;
                    const int32_t du = (int32_t)(bits(got) - bits(want));
                    worse += du > 1 || du < -1;
                }
            }
        }
        printf("div_in_range: %ld cases (reciprocal estimate off by -2..+2 ulp), %ld not the IEEE quotient (%.2e), %ld off by more than an ulp\n",
               n, bad, (double)bad / n, worse);
        fail |= worse != 0 || bad * 10000 > n;
    }

    // ---- 2. one-pole k = e^-theta
    {
        std::mt19937_64 rng(99);
        double worst = 0.0;
        const long N = quick ? 400000 : 4000000;
        for (long i = 0; i < N; i++) {
            const double u = (rng() >> 11) * (1.0 / 9007199254740992.0);
            const float th = (float)(0.004 * exp(u * log(40.0 / 0.004)));
            const float k = exp_neg_fast<float>(th);
            const double want = exp(-(double)th);
            const double ulp = (double)(fbits(bits((float)want) + 1u) - (float)want);
            const double e = fabs((double)k - want) / ulp;
            if (e > worst) worst = e;
        }
        printf("exp_neg_fast: worst error %.2f ulp over theta in [0.004, 40] (host exp2f standing in for ex2.approx)\n", worst);
        fail |= worst > 4.0;
    }

    // ---- 2b. exp_neg_fast at an overflowing cutoff: theta = +inf gives k = 0 (the reference's exp(-inf)), and the
    //          clamp that does it changes no other result: below kThetaBig every binary32 theta keeps the bits of the
    //          unclamped form; from kThetaBig up, the unclamped form gave 0, or NaN once theta * log2 e overflows
    {
        auto unclamped = [](float th) {
            const float L1 = 0x1.715476p+0f, L2 = 0x1.4ae0c0p-26f;
            const float tn = th * -L1;
            const float r = fmaf(th, L1, tn);
            const float tl = fmaf(th, L2, r);
            const float e = vex2(tn);
            return fmaf(e, tl * -0x1.62e430p-1f, e);
        };
        const float inf = INFINITY;
        const float kinf = exp_neg_fast<float>(inf);
        long n = 0, changed = 0, bad_big = 0;
        const uint32_t step = quick ? 61u : 1u;
        for (uint64_t u = 0; u <= 0xffffffffull; u += step) {
            const float th = fbits((uint32_t)u);
            if (th != th) continue;                                         // NaN: not an angle
            const float got = exp_neg_fast<float>(th), old = unclamped(th);
            n++;
            if (th < kThetaBig) {
                changed += bits(got) != bits(old);
            } else {
                const bool old_ok = bits(old) == 0u || (old != old && std::isinf(th * 0x1.715476p+0f));
                bad_big += bits(got) != 0u || !old_ok;
            }
        }
        printf("exp_neg_fast clamp: k(+inf) = %g; %ld thetas, %ld below %g changed, %ld from it up not (k = 0, was 0 "
               "or NaN)\n", (double)kinf, n, changed, (double)kThetaBig, bad_big);
        fail |= bits(kinf) != 0u || changed != 0 || bad_big != 0;
    }

    // ---- 3. windows.  "slack" = |result - exact| - ulp(result)/2: what the evaluation adds on top of a correct rounding.
    for (int pass = 0; pass < 2; pass++) {
        // pass 0: sweeps as slow as the bench bank's (|d| <= 2 % of theta); pass 1: anything a valid window admits
        std::mt19937_64 rng(777);
        long n = 0, bs = 0, bc = 0;
        double ws = 0, wc = 0;
        const long N = quick ? 200000 : 2000000;
        for (long i = 0; i < N; i++) {
            const double u = (rng() >> 11) * (1.0 / 9007199254740992.0);
            const float thc = (float)(0.004 * exp(u * log(3.1 / 0.004)));              // log-uniform 0.004 .. 3.1
            Window W;
            make_window(W, thc);
            for (int j = 0; j < 16; j++) {
                const double v = (rng() >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
                const float lim = thc * (pass == 0 ? 0.02f : 0.5f);
                const float dmax = lim < kWinDelta ? lim : kWinDelta;
                const float th = thc + (float)(v * dmax);
                float s, c;
                window_sincos<float>(W, th - thc, &s, &c);                 // exact difference (Sterbenz)
                const double sd = sin((double)th), cd = cos((double)th);
                n++;
                bs += bits(s) != bits((float)sd); bc += bits(c) != bits((float)cd);
                auto slack = [](float got, double want) {
                    const double half_ulp = 0.5 * (double)(fbits(bits(fabsf(got)) + 1u) - fabsf(got));
                    const double x = fabs((double)got - want) - half_ulp;
                    return x > 0.0 ? x : 0.0;
                };
                const double es = slack(s, sd), ec = slack(c, cd);
                if (es > ws) ws = es;
                if (ec > wc) wc = ec;
            }
        }
        printf("windows (%s): %ld frames; != rounded-once: sin %.3f%% cos %.3f%%; worst slack beyond a correct "
               "rounding: sin %.1e cos %.1e\n", pass == 0 ? "|d| <= 2% of theta" : "|d| <= 50% of theta, 2^-7",
               n, 100.0 * bs / n, 100.0 * bc / n, ws, wc);
        fail |= ws > 4e-9 || wc > 4e-9;
        if (pass == 0) fail |= bs > n / 50 || bc > n / 50;
    }

    // ---- 4. theta = (2 pi fl) / sr
    {
        const float rates[] = {8000.0f, 16000.0f, 22050.0f, 32000.0f, 44100.0f, 48000.0f, 88200.0f, 96000.0f, 192000.0f};
        long bad = 0, n = 0;
        for (float sr : rates) {
            const float rsr = 1.0f / sr;
            // fl from 2^-20 Hz up to where theta passes 4 (beyond any valid window); every binary32 in between
            const uint32_t lo = bits(0x1p-20f), hi = bits(4.0f * sr / kTwoPi);
            const uint32_t step = quick ? 7u : 1u;
            for (uint32_t u = lo; u <= hi; u += step) {
                const float fl = fbits(u);
                const float want = (fl * kTwoPi) / sr;
                const float got = theta_of<float>(fl, sr, rsr);
                n++;
                bad += bits(got) != bits(want);
            }
        }
        printf("theta_of: %ld numerators at 9 sample rates, %ld not the IEEE quotient\n", n, bad);
        fail |= bad != 0;
    }

    // ---- 5. 2^x around a window's centre
    {
        std::mt19937_64 rng(4242);
        long n = 0, bad = 0, worse = 0;
        const long N = quick ? 200000 : 2000000;
        for (long i = 0; i < N; i++) {
            const double u = (rng() >> 11) * (1.0 / 9007199254740992.0);
            Window W;
            W.xc = (float)(u * 24.0 - 12.0);
            split_hi_rel(s2_exp2_d(W.xc), &W.Eh, &W.Er);
            for (int j = 0; j < 16; j++) {
                const double v = (rng() >> 11) * (1.0 / 9007199254740992.0) * 2.0 - 1.0;
                const float x = W.xc + (float)(v * kWinDeltaX);
                const float got = sweep_exact<float>(W, x, 1.0f);
                const float want = s2_exp2f(x);
                n++;
                if (bits(got) != bits(want)) {
                    bad++;
                    const int32_t du = (int32_t)(bits(got) - bits(want));
                    worse += du > 1 || du < -1;
                }
            }
        }
        printf("sweep_exact: %ld arguments, %ld not 2^x rounded once (%.3f%%), %ld off by more than an ulp\n",
               n, bad, 100.0 * bad / n, worse);
        fail |= worse != 0 || bad * 100 > n;
    }

    // ---- 6. a decay sweep at the worst corner: cutoff 100..200 Hz, damping 0.2, 1.5 octaves over 9600 frames
    {
        const float sr = 48000.0f, rsr = 1.0f / sr, one = 1.0f, hd = 0.1f, amt = 1.5f;
        double worst_out = 0.0;
        long coef_diff = 0, frames = 0;
        for (int voice = 0; voice < (quick ? 8 : 64); voice++) {
            const float lpf = 100.0f + 1.7f * (float)voice;
            const float P = sr / (55.0f * (1.0f + 0.37f * (float)voice));
            const float A = 0.0f, D = 9600.0f, sD = (0.0f - 1.0f) / D;
            float ph = 0.0f;
            float xa1 = 0, xa2 = 0, ya1 = 0, ya2 = 0, xb1 = 0, xb2 = 0, yb1 = 0, yb2 = 0;
            Window W; W.k = 0xffffffffu;
            for (uint32_t n = 0; n < 9600; n++) {
                const float x = (float)n;
                const float m = (sD * (x - A)) + 1.0f;
                if ((n >> 5) != W.k) {
                    const float xc = (float)((n & ~31u) + 16u);
                    W.xc = ((sD * (xc - A)) + 1.0f) * amt;
                    const double Ed = s2_exp2_d(W.xc);
                    split_hi_rel(Ed, &W.Eh, &W.Er);
                    make_window(W, (((float)Ed * lpf) * kTwoPi) / sr);
                    W.k = n >> 5;
                }
                float s, c, a0, a1, a2, b0, b1, b2;
                const float E = sweep_exact<float>(W, m * amt, one);
                window_sincos<float>(W, theta_of<float>(E * lpf, sr, rsr) - W.thc, &s, &c);
                biquad_lp_hp<false, float>(s, c, hd, one, &a0, &a1, &a2);
                // the full evaluation: the reference's chain (process.rs:244-246, dsp_filters.rs:99-109)
                const float th = ((s2_exp2f(m * amt) * lpf) * kTwoPi) / sr;
                float sf, cf; s2_sincosf(th, &sf, &cf);
                biquad_lp_hp_any<false>(sf, cf, hd, one, &b0, &b1, &b2);
                coef_diff += bits(a0) != bits(b0) || bits(a1) != bits(b1) || bits(a2) != bits(b2);
                frames++;
                // saw + 1 (the x16 path's input, process.rs:341-345), both filters (dsp_filters.rs:116-128)
                const float u = (1.0f - 2.0f * ph) + 1.0f;
                ph += 1.0f / P; if (ph >= 1.0f) ph -= 1.0f;
                float sx = (u + 2.0f * xa1) + xa2;
                float t = a0 * sx; t = t + a2 * ya1; t = t - a1 * ya2;
                xa2 = xa1; xa1 = u; ya2 = ya1; ya1 = t;
                sx = (u + 2.0f * xb1) + xb2;
                float w = b0 * sx; w = w + b2 * yb1; w = w - b1 * yb2;
                xb2 = xb1; xb1 = u; yb2 = yb1; yb1 = w;
                const double dv = fabs((double)t - (double)w);
                if (dv > worst_out) worst_out = dv;
            }
        }
        printf("decay sweep: %ld frames, %ld with a coefficient differing from the full evaluation (%.3f%%), worst output "
               "difference %.2e\n", frames, coef_diff, 100.0 * coef_diff / frames, worst_out);
        // (one differing ulp in one frame is enough to decorrelate the two filters' rounding, after which they sit
        // apart by the binary32 direct form's own noise floor at this corner, ~5e-5 rms: the output difference is
        // reported, the coefficient mismatch rate is what is asserted — glibc's sinf / cosf, which the oracle
        // calls, differ from the rounded-once values in 1.3 % of arguments)
        fail |= coef_diff * 50 > frames;
    }
    printf(fail ? "FAILED\n" : "ok\n");
    return fail;
}
