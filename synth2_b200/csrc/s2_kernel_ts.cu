// s2_kernel_ts.cu — time-split rendering for narrow banks (BASELINE config 2: 1,024 voices x 4,096 frames).
//
// A bank of a thousand voices is 32 warps: with one voice per lane the whole GPU waits on 32 dependent
// instruction streams (131 us per 16 MiB block, 2 % of the HBM roofline).  Voices are independent but so,
// almost, are the time segments of one voice: everything in a frame is a closed form of the frame offset
// except the two recurrences —
//
//   * the oscillator phase, phase' = (phase + 1/P) % 1 in binary32 (try3/oscillators.rs:377-381), whose
//     rounding cannot be reassociated if it is to stay bit-exact: it is stepped sequentially, but ALONE
//     (3 dependent instructions per frame instead of the whole frame), by `ts_phase_kernel`, which records
//     the phase at the start of each of the block's 32 time segments;
//   * the filter, an affine map of its state.  One-pole y = fma(1-k, u, k*y') (try3/filters.rs:15-34): segment
//     s as a whole is y_out = K*y_in + Y_s with K = k^L and Y_s its zero-state response.  Second-order low-pass
//     (try3/dsp_filters.rs:116-128): the recursive state is Y = (y1, y2), one frame is Y' = M Y + (2a*s, 0)
//     with M = [[2g, -2b], [1, 0]], so a segment is Y_out = M^L Y_in + Z_s (the delayed inputs x1, x2 are not
//     state to be scanned: they are the oscillator + noise of the two frames before the segment, recomputed
//     from their recorded phases).  The 32 segment maps of a voice compose by a warp-shuffle prefix scan (the
//     "parallel prefix scan over the associative affine / 2x2 state-transition operator" of the north star).
//
// `ts_render_kernel`: one warp per voice, lane s = frames [s*L, (s+1)*L) of the block (L = frames / 32).
// Sweep 1 renders the segment from a zero filter state to get Y_s; the scan gives every lane its true start
// state; sweep 2 renders the segment again from that state with the reference's own recurrence and writes
// it out through the transposed smem tile (128-byte runs per row, like the wide-bank kernel).  The second
// sweep costs nothing that matters: the shape is latency-bound and the machine is otherwise idle.
//
// Parity: phase bit-exact (same recurrence, same order); output within the north-star tolerance (the start
// state of segments 1..31 carries the scan's reassociation error, ~1 ulp of the state, and decays as k^n).
// Used only when every voice of the block has a constant period (host check in s2_capi.cu: no pitch modulation);
// anything else renders through the wide-bank kernel.  Where a cutoff follows a ramping mod envelope the sweeps
// evaluate the coefficients per frame (ts_moving_sweep) and the segment map is the product of the per-frame maps.
#include "s2_device.cuh"

namespace s2 {
namespace {

constexpr int kSegs = 32;                 // time segments per block = lanes per warp

// K1: lane = voice slot.  phase recurrence only, 8 frames per trip.
__global__ void __launch_bounds__(32) ts_phase_kernel(const RenderArgs a, float* __restrict__ seg_phase) {
    const uint32_t slot = blockIdx.x * 32u + threadIdx.x;
    if (slot >= a.slot_end) return;
    const uint32_t vp = a.vpad;
    const float* __restrict__ P = a.params + slot;
    if (__float_as_uint(P[P_ACTIVE * vp]) == 0u) return;
    float* __restrict__ S = a.state + slot;
    OscC oc;
    make_osc(oc, P[P_PITCH * vp], a.sample_rate);            // mod_env_to_osc_freq == 0: fo == pitch exactly
    const float d = oc.d;
    float ph = __float_as_uint(S[S_HAS_PHASE * vp]) != 0u ? S[S_PHASE * vp] : 0.0f;      // process.rs:316
    const uint32_t L = a.frames / kSegs;
    // seg_phase[slot][plane][segment]: plane 0 = phase of the segment's first frame, planes 1 / 2 = phase of the
    // one / two frames before it (the biquad's delayed inputs are recomputed from them)
    float* __restrict__ out = seg_phase + (size_t)slot * (3 * kSegs);
    float p1 = 0.0f, p2 = 0.0f;
    for (int s = 0; s < kSegs; s++) {
        out[s] = ph;
        out[kSegs + s] = p1;
        out[2 * kSegs + s] = p2;
#pragma unroll 1
        for (uint32_t j = 0; j < L; j += 8u) {
            const bool last = j + 8u == L;
#pragma unroll
            for (int i = 0; i < 8; i++) {
                if (i == 6) p2 = last ? ph : p2;
                if (i == 7) p1 = last ? ph : p1;
                ph = wrap_unit(__fadd_rn(ph, d));            // fmod(phase + d, 1), s2_device.cuh
            }
        }
    }
    S[S_PHASE * vp] = ph;
    S[S_HAS_PHASE * vp] = __uint_as_float(1u);
}

template <int FILTER, bool GCONST>
__device__ __forceinline__ void ts_chunk_kind(FastV& F, const EnvQ* amp, float one, uint32_t kind, uint32_t rot, uint32_t n,
                                              float* row, const float* sintab) {
    constexpr int G = GCONST ? G_CONST : G_ANY;
    // warp-uniform: a warp is one voice
    with_kind<0, 1, 2, 3>((int)kind, [](auto K, auto&&... args) { chunk_fast_tp<FILTER, K, G, false, TRACE_NONE>(args...); },
                          F, amp, one, kind, rot, n, row, sintab);
}

// Write-back of the 32 x 32 tile of frames c .. c + 31 of every segment: tile row r = segment r (128-byte runs)
__device__ __forceinline__ void ts_store_tile(const float* tile, int lane, float* __restrict__ gout, uint32_t L, uint32_t c) {
    const int q = lane >> 3, c4 = (lane & 7) * 4;
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const int r = 4 * i + q;
        const float4 val = *reinterpret_cast<const float4*>(tile + r * kTsTileStride + c4);
        __stcs(reinterpret_cast<float4*>(gout + (size_t)r * L + c + c4), val);
    }
    __syncwarp();
}

// 2x2 real matrices (row-major) in binary64 for the biquad's segment maps
struct M22 { double a, b, c, d; };
__device__ __forceinline__ M22 mul(const M22& x, const M22& y) {       // x * y
    return {fma(x.a, y.a, x.b * y.c), fma(x.a, y.b, x.b * y.d), fma(x.c, y.a, x.d * y.c), fma(x.c, y.b, x.d * y.d)};
}
__device__ __forceinline__ M22 shfl_up(const M22& m, int off) {
    return {__shfl_up_sync(0xffffffffu, m.a, off), __shfl_up_sync(0xffffffffu, m.b, off),
            __shfl_up_sync(0xffffffffu, m.c, off), __shfl_up_sync(0xffffffffu, m.d, off)};
}

// One sweep over a lane's segment with a MOVING cutoff (the mod envelope is in a ramp: the first 200 ms of every
// note of the default patch).  Per frame, exactly the per-frame functions of the wide-bank kernel (x16_coefs:
// envelopes by stage line, the moving or resting coefficient evaluation, oscillator, noise, filter step); the first sweep also
// accumulates the product of the per-frame state maps — k_n for the one-pole, M_n = [[2g_n, -2b_n], [1, 0]] for
// the biquad — which is the segment's map for the scan.  WRITE: second sweep, output through the tile.
template <int FILTER, bool WRITE>
__device__ __forceinline__ void ts_moving_sweep(FastV& F, const Lane& V, float sr, float one, uint32_t nl, uint32_t L,
                                                float& kprod, M22& mprod, float* tile, int lane, float* __restrict__ gout,
                                                const float* sintab) {
    float* row = tile + lane * kTsTileStride;
    SegEnv sa = seg_env(V.amp, nl);
    uint32_t n = nl;
    float xf = __uint2float_rn(nl);
    FiltC fc;
    fc.c0 = fc.c1 = fc.c2 = 0.0f; fc.fl_bits = kNoKey;
    MovG mg;
    movg_init(mg, V.lpf, V.amt_lpf, V.damp, sr);
    mg.sm = seg_env(V.mod, nl);
    for (uint32_t c = 0; c < L; c += kChunk) {
#pragma unroll 1
        for (int i = 0; i < kChunk; i++) {
            if (n >= mg.sm.nend) mg.sm = seg_env(V.mod, n);
            const float m = seg_eval(mg.sm, xf);
            x16_coefs<FILTER>(fc, mg, V.mod, V.lpf, V.amt_lpf, V.damp, sr, one, n, m);
            const float y = voice_frame<FILTER, -1>(F, fc, V.kind, V.rot, n, sintab);
            if (!WRITE) {
                if (FILTER == 0) kprod = __fmul_rn(kprod, fc.c0);
                else {                                        // M_n * mprod
                    const double g2 = (double)fc.c2, b2 = (double)fc.c1;
                    const M22 t = {fma(g2, mprod.a, -b2 * mprod.c), fma(g2, mprod.b, -b2 * mprod.d), mprod.a, mprod.b};
                    mprod = t;
                }
            } else {
                row[i] = __fmul_rn(y, seg_walk(sa, V.amp, n, xf));
            }
            n += 1u;
            xf = __fadd_rn(xf, 1.0f);
        }
        if (WRITE) ts_store_tile(tile, lane, gout, L, c);
    }
}

// K2: one warp per voice slot; lane = time segment.
template <int FILTER, bool MOVING>
__global__ void __launch_bounds__(32) ts_render_kernel(const RenderArgs a, const float* __restrict__ seg_phase) {
    extern __shared__ __align__(16) float smem[];
    float* tile = smem;                                      // [32 segments][kTsTileStride]
    float* sintab = smem + 32 * kTsTileStride;
    const int lane = threadIdx.x;
    const uint32_t slot = blockIdx.x;
    const uint32_t vp = a.vpad;
    const float sr = a.sample_rate;
    const float* __restrict__ P = a.params + slot;           // warp-uniform loads
    const uint32_t frames = a.frames;
    const uint32_t L = frames / kSegs;
    const uint32_t orow = __float_as_uint(P[P_ROW * vp]);
    if (orow == kPadRow) return;                             // a padding slot of a routed bank: no voice, no row
    float* __restrict__ gout = a.voice_out + (size_t)orow * a.row_stride;

    if (__float_as_uint(P[P_ACTIVE * vp]) == 0u) {
        // inactive voices render silence (their state does not move)
        for (uint32_t t = (uint32_t)lane * 4u; t < frames; t += 128u)
            __stcs(reinterpret_cast<float4*>(gout + t), make_float4(0.0f, 0.0f, 0.0f, 0.0f));
        return;
    }
    const Lane V = load_lane(P, vp, sr, __float_as_uint(P[P_RELEASE * vp]));
    const uint32_t kind = V.kind, rot = V.rot;
    if (kind == 3u) {
        for (int i = lane; i < 1024; i += 32) sintab[i] = __uint_as_float(d_sin_bits[i]);
    }
    const EnvQ Aq = compact(V.amp);
    float* __restrict__ S = a.state + slot;
    const uint32_t n0 = __float_as_uint(S[S_OFFSET * vp]);

    // constants of the block: the host admitted this voice because its period and cutoff do not move
    const float m = (V.amt_lpf != 0.0f && env_stage(V.mod, __uint2float_rn(n0)) == 2) ? V.mod.S : 0.0f;
    const float fl = modulate_freq(V.lpf, m, V.amt_lpf);
    OscC oc;
    FiltC fc;
    make_osc(oc, V.pitch, sr);
    make_filt<FILTER>(fc, fl, V.damp, sr);

    FastV F;
    set_osc(F, oc);
    F.gain = V.gain; F.namt = V.namt;
    F.fc = fc;
    F.es = 0.0f; F.nex0 = 0.0f; F.ey0 = 1.0f; F.seg_end = 0u;
    const float* __restrict__ sp = seg_phase + (size_t)slot * (3 * kSegs);
    const float ph0 = sp[lane];
    const uint32_t nl = n0 + (uint32_t)lane * L;             // this lane's first frame offset
    float* row = tile + lane * kTsTileStride;
    __syncwarp();

    // delayed inputs of the biquad at the segment start: carried state for segment 0, otherwise the
    // oscillator + noise of the two frames before the segment (process.rs:341-358 on their recorded phases)
    float x1_in = 0.0f, x2_in = 0.0f;
    if (FILTER == 1) {
        if (lane == 0) { x1_in = S[S_X1 * vp]; x2_in = S[S_X2 * vp]; }
        else {
            float pa = sp[kSegs + lane], pb = sp[2 * kSegs + lane];
            const float oa = osc_step<-1, false>(kind, oc, pa, sintab);
            const float ob = osc_step<-1, false>(kind, oc, pb, sintab);
            x1_in = input1(F, oa, rot, nl - 1u);
            x2_in = input1(F, ob, rot, nl - 2u);
        }
    }

    // ---- sweep 1: zero-state response of the segment (gain and output are irrelevant)
    float kprod = 1.0f;
    M22 mprod = {1.0, 0.0, 0.0, 1.0};
    F.ph = ph0;
    F.fs = {x1_in, x2_in, 0.0f, 0.0f};
    if (MOVING) {
        ts_moving_sweep<FILTER, false>(F, V, sr, a.one, nl, L, kprod, mprod, tile, lane, gout, sintab);
    } else {
        for (uint32_t c = 0; c < L; c += kChunk) ts_chunk_kind<FILTER, true>(F, &Aq, a.one, kind, rot, nl + c, row, sintab);
    }

    // ---- the segment maps compose left to right: inclusive Hillis-Steele scan over the lanes
    float y1_in, y2_in = 0.0f;
    if (FILTER == 0) {
        const float last = S[S_LAST * vp];
        float Kc = MOVING ? kprod : (float)exp((double)L * log((double)fc.c0));   // k^L (one value per voice)
        float Yc = F.fs.y1;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const float Kp = __shfl_up_sync(0xffffffffu, Kc, off);
            const float Yp = __shfl_up_sync(0xffffffffu, Yc, off);
            if (lane >= off) {                                // (Kp, Yp) happens first, then (Kc, Yc)
                Yc = __fmaf_rn(Kc, Yp, Yc);
                Kc = __fmul_rn(Kc, Kp);
            }
        }
        const float end_state = __fmaf_rn(Kc, last, Yc);      // state after this lane's segment
        y1_in = __shfl_up_sync(0xffffffffu, end_state, 1);
        if (lane == 0) y1_in = last;
    } else {
        // one frame: (y1, y2)' = M (y1, y2) + (2a*s, 0),  M = [[2g, -2b], [1, 0]]  (filt_step<1>)
        M22 Mc = mprod;
        if (!MOVING) {
            M22 base = {(double)fc.c2, -(double)fc.c1, 1.0, 0.0};
            for (uint32_t e = L; e; e >>= 1) {                // M^L by squaring
                if (e & 1u) Mc = mul(base, Mc);
                base = mul(base, base);
            }
        }
        double z1 = (double)F.fs.y1, z2 = (double)F.fs.y2;          // zero-state response of this segment
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const M22 Mp = shfl_up(Mc, off);
            const double p1 = __shfl_up_sync(0xffffffffu, z1, off), p2 = __shfl_up_sync(0xffffffffu, z2, off);
            if (lane >= off) {                                // earlier map (Mp, p) first, then (Mc, z)
                const double n1 = fma(Mc.a, p1, fma(Mc.b, p2, z1));
                const double n2 = fma(Mc.c, p1, fma(Mc.d, p2, z2));
                z1 = n1; z2 = n2;
                Mc = mul(Mc, Mp);
            }
        }
        const double y10 = (double)S[S_Y1 * vp], y20 = (double)S[S_Y2 * vp];
        const double e1 = fma(Mc.a, y10, fma(Mc.b, y20, z1));    // state after this lane's segment
        const double e2 = fma(Mc.c, y10, fma(Mc.d, y20, z2));
        const double u1 = __shfl_up_sync(0xffffffffu, e1, 1), u2 = __shfl_up_sync(0xffffffffu, e2, 1);
        y1_in = lane == 0 ? (float)y10 : (float)u1;
        y2_in = lane == 0 ? (float)y20 : (float)u2;
    }

    // ---- sweep 2: the reference recurrence from the true start state, written out
    F.ph = ph0;
    F.fs = {x1_in, x2_in, y1_in, y2_in};
    if (MOVING) {
        ts_moving_sweep<FILTER, true>(F, V, sr, a.one, nl, L, kprod, mprod, tile, lane, gout, sintab);
    } else {
        for (uint32_t c = 0; c < L; c += kChunk) {
            ts_chunk_kind<FILTER, false>(F, &Aq, a.one, kind, rot, nl + c, row, sintab);
            ts_store_tile(tile, lane, gout, L, c);
        }
    }
    if (lane == 31) {
        if (FILTER == 0) S[S_LAST * vp] = F.fs.y1;
        else { S[S_X1 * vp] = F.fs.x1; S[S_X2 * vp] = F.fs.x2; S[S_Y1 * vp] = F.fs.y1; S[S_Y2 * vp] = F.fs.y2; }
        S[S_OFFSET * vp] = __uint_as_float(n0 + frames);      // n0 + frames <= 2^24 (host check)
    }
}

// The mix of a bank of at most one warp's voices, in the reference's order (synth.rs:176-202): one thread per frame
// adds the rows in voice order to an accumulator that starts at +0.0, so a lone -0.0 sample comes out as +0.0.
__global__ void __launch_bounds__(256) ts_mix_rows_kernel(const float* __restrict__ rows, uint32_t n_rows,
                                                          size_t row_stride, uint32_t frames, float* __restrict__ bus) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= frames) return;
    float acc = 0.0f;
    for (uint32_t r = 0; r < n_rows; r++) acc = __fadd_rn(acc, rows[(size_t)r * row_stride + t]);
    bus[t] = acc;
}

}  // namespace

cudaError_t launch_ts_mix_rows(const float* rows, uint32_t n_rows, size_t row_stride, uint32_t frames, float* bus,
                               cudaStream_t stream) {
    if (frames == 0) return cudaSuccess;
    ts_mix_rows_kernel<<<(frames + 255u) / 256u, 256, 0, stream>>>(rows, n_rows, row_stride, frames, bus);
    return cudaGetLastError();
}

cudaError_t launch_ts_phase(const RenderArgs& a, float* seg_phase, cudaStream_t stream) {
    if (a.slot_end == 0) return cudaSuccess;
    ts_phase_kernel<<<(a.slot_end + 31u) / 32u, 32, 0, stream>>>(a, seg_phase);
    return cudaGetLastError();
}

cudaError_t launch_ts_render(const RenderArgs& a, uint32_t filter_kind, bool moving, const float* seg_phase,
                             cudaStream_t stream) {
    if (a.slot_end == 0) return cudaSuccess;
    const size_t smem = (32 * kTsTileStride + 1024) * sizeof(float);
    if (filter_kind == 0) {
        if (moving) ts_render_kernel<0, true><<<a.slot_end, 32, smem, stream>>>(a, seg_phase);
        else ts_render_kernel<0, false><<<a.slot_end, 32, smem, stream>>>(a, seg_phase);
    } else {
        if (moving) ts_render_kernel<1, true><<<a.slot_end, 32, smem, stream>>>(a, seg_phase);
        else ts_render_kernel<1, false><<<a.slot_end, 32, smem, stream>>>(a, seg_phase);
    }
    return cudaGetLastError();
}

}  // namespace s2
