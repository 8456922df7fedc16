// s2_kernels.cu — sm_100a render kernels for synth2's oscillator -> filter -> envelope -> mix path.
//
// Mapping (DESIGN.md section 4): one lane = one voice, one warp = 32 consecutive voice slots, time runs
// sequentially inside the lane (the f32 phase recurrence of oscillators.rs:377-381 is not
// associative, so its rounding sequence is replayed exactly).  A warp produces a 32 voices x 32
// frames tile in shared memory and writes it back transposed, so every STG.128 of the warp
// covers four full 128-byte lines of voice-major output.
//
// Arithmetic contract: every operation below that feeds a discrete decision (phase, table index,
// envelope stage, noise hash) is the reference's binary32 operation, spelled with __f*_rn
// intrinsics so nothing is contracted or reassociated (the file is also built with -fmad=false).
// Reference line numbers are relative to /root/reference/components/s2_lib/src/.
#include "s2_device.cuh"

// Register cap of the render kernel, as a minimum of resident one-warp blocks per SM: 16 blocks = 65,536 / (16 * 32)
// = 128 registers.  Shared memory (14.8 KB + 1 KB per block) already limits an SM to 14 blocks — the 13.8 a
// 65,536-voice bank needs — so nothing is lost against the 96 registers of round 1, and the chunk-level state
// (classification counters, tile pointers) no longer spills around the inlined loops: the spill reloads sat at
// the head of every chunk and showed as long-scoreboard stalls (21 % of the samples of a moving-cutoff launch).
#ifndef S2_MINBLOCKS
#define S2_MINBLOCKS 16
#endif

namespace s2 {

// Sum of a lane's N float4 tile reads as a pairwise tree of packed adds (depth log2 N instead of a chain of
// N: the adds sit at the end of a chunk where the warp has nothing else to issue).  Fixed order: deterministic.
template <int N>
__device__ __forceinline__ void tree_sum_rows(float4 (&val)[N], float2& b01, float2& b23) {
#pragma unroll
    for (int w = 1; w < N; w <<= 1) {
#pragma unroll
        for (int i = 0; i + w < N; i += 2 * w) {
            const float2 lo = padd2(make_float2(val[i].x, val[i].y), make_float2(val[i + w].x, val[i + w].y));
            const float2 hi = padd2(make_float2(val[i].z, val[i].w), make_float2(val[i + w].z, val[i + w].w));
            val[i] = make_float4(lo.x, lo.y, hi.x, hi.y);
        }
    }
    b01 = make_float2(val[0].x, val[0].y);
    b23 = make_float2(val[0].z, val[0].w);
}

// Shared memory of a metered launch (TRACE_METER), after the warp's tiles: each lane's running meters, double
// sum_sq[32] then uint32 peak[32].  Kept there rather than in registers, which the chunk loops use up to the cap.
constexpr int kMeterFloats = 32 * 2 + 32;
__device__ __forceinline__ double* meter_sum(float* smem) { return reinterpret_cast<double*>(smem + warp_smem_floats()); }
__device__ __forceinline__ uint32_t* meter_peak(float* smem) { return reinterpret_cast<uint32_t*>(smem + warp_smem_floats() + 64); }

// Meters of one 64-frame tile row (the lane's own): squares in binary32, summed by a fixed pairwise tree over the 64
// columns counted from the tile's first frame, the tile total added to the binary64 running total; the peak is the
// largest magnitude as bits (sign cleared), so a NaN ranks above +inf.  A partial tile zeroes its columns from `cnt`
// on first (other lanes read only the first `cnt`).  One tree for every tile of every write-back: the total's bits
// do not depend on whether rows or a bus are stored.
__device__ __forceinline__ void meter_row(float* row, uint32_t cnt, float one, double& sum_sq, uint32_t& peak) {
    if (cnt < (uint32_t)kTileFrames)
        for (uint32_t c = cnt; c < (uint32_t)kTileFrames; c++) row[c] = 0.0f;
    constexpr uint32_t m = 0x7fffffffu;
    uint32_t pk = peak;
    float2 half[2];
#pragma unroll
    for (int hh = 0; hh < 2; hh++) {
        float2 s[16];
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const float4 v = *reinterpret_cast<const float4*>(row + 32 * hh + 4 * i);
            s[2 * i] = pmul2(make_float2(v.x, v.y), make_float2(v.x, v.y));
            s[2 * i + 1] = pmul2(make_float2(v.z, v.w), make_float2(v.z, v.w));
            pk = __vimax3_u32(pk, __float_as_uint(v.x) & m, __float_as_uint(v.y) & m);
            pk = __vimax3_u32(pk, __float_as_uint(v.z) & m, __float_as_uint(v.w) & m);
        }
        // the first level adds two products: vaddp, which ptxas cannot fuse with the multiplies (s2_cutoff.h)
#pragma unroll
        for (int i = 0; i < 16; i += 2) s[i] = s2c::vaddp(s[i], s[i + 1], one);
#pragma unroll
        for (int w = 2; w < 16; w <<= 1)
#pragma unroll
            for (int i = 0; i + w < 16; i += 2 * w) s[i] = padd2(s[i], s[i + w]);
        half[hh] = s[0];
    }
    const float2 t = padd2(half[0], half[1]);
    sum_sq = __dadd_rn(sum_sq, (double)__fadd_rn(t.x, t.y));
    peak = pk;
}

// One fast chunk of a kind-uniform (or mixed, KIND = -1) warp, by envelope mode and hash form.
// Instruction-cache budget: an SM holds 32 KB of instructions (L1.5; 6 KB per scheduler in L0) and its warps sit in
// different loops (two oscillator kinds x envelope modes); once the loops in flight plus the per-chunk code outgrow
// that, warps stall on instruction fetch at each 128-byte line (profiles/r2_notes.md).  So the rare chunk that
// holds a stage boundary does not get a specialised loop per kind: it goes through the compact per-frame loop
// (chunk_modcut_sc with a resting cutoff), ~1 KB shared by all kinds.
template <int FILTER, int KIND, int TRACE>
__device__ __forceinline__ void fast_tile(int gmode, bool fasthash, FastV& F, const EnvQ* amp, float one, uint32_t kind,
                                          uint32_t rot, uint32_t n, float* row, const float* sintab) {
    if (!fasthash) {
        // banks with added noise amounts or odd offsets: one general variant per kind is their whole hot path
        chunk_fast_tp<FILTER, KIND, G_ANY, false, TRACE>(F, amp, one, kind, rot, n, row, sintab);
    } else if (gmode == G_CONST) {
        chunk_fast_tp<FILTER, KIND, G_CONST, true, TRACE>(F, amp, one, kind, rot, n, row, sintab);
    } else {
        chunk_fast_tp<FILTER, KIND, G_LINE, true, TRACE>(F, amp, one, kind, rot, n, row, sintab);
    }
}

// One warp renders 32 consecutive slots; lane l owns slot base + l.
// 65,536 voices = 13.8 one-warp blocks per SM: without pipelining all of them must be resident at once (a
// second wave would serialise: measured +20 % time at 144 registers, where only 13 fit).
template <int FILTER, int TRACE>
__global__ void __launch_bounds__(32, S2_MINBLOCKS)
render_kernel(const RenderArgs a) {
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x;
    constexpr int kRows = 32;
    float* tile = smem;
    float* cold_base = smem + kRows * kTileStride;
    constexpr bool kMeter = TRACE == TRACE_METER;
    float* sintab = smem + warp_smem_floats() + (kMeter ? kMeterFloats : 0);
    if constexpr (kMeter) {
        meter_sum(smem)[lane] = 0.0;
        meter_peak(smem)[lane] = 0u;
    }
    if (a.has_sine) {
        for (int i = lane; i < 1024; i += 32) sintab[i] = __uint_as_float(d_sin_bits[i]);
        __syncthreads();
    }

    const uint32_t vbase = a.slot_begin + blockIdx.x * kRows;
    if (vbase >= a.slot_end) return;
    const uint32_t vp = a.vpad;
    const float sr = a.sample_rate;
    const float rsr = __frcp_rn(sr);
    const float one = a.one;
    Cold& C = *reinterpret_cast<Cold*>(cold_base + lane * kColdWords);
    float* row = tile + lane * kTileStride;

    uint32_t kind, rot, n;
    bool active;
    FastV F{};
    {
        const uint32_t v = vbase + lane;
        const bool exists = v < a.slot_end;
        const uint32_t vi = exists ? v : vbase;    // out-of-range lanes shadow slot vbase's loads, never store
        const float* __restrict__ P = a.params + vi;
        active = exists && __float_as_uint(P[P_ACTIVE * vp]) != 0u;
        C.vi = vi;
        C.out_row = exists ? __float_as_uint(P[P_ROW * vp]) : 0xffffffffu;
        uint32_t release = __float_as_uint(P[P_RELEASE * vp]);
        if (a.staged_release != nullptr && exists) {
            release = a.staged_release[C.out_row];
            a.release_row[vi] = release;
        }
        C.release = release;
        const Lane L = load_lane(P, vp, sr, release);
        kind = L.kind;
        rot = L.rot;
        C.amp = compact(L.amp);
        C.mod = compact(L.mod);
        C.pitch = L.pitch; C.lpf = L.lpf; C.damp = L.damp; C.amt_osc = L.amt_osc; C.amt_lpf = L.amt_lpf;
        C.flags = (active ? 1u : 0u) | ((L.amt_osc != 0.0f || L.amt_lpf != 0.0f) ? 2u : 0u);
        C.theta0 = theta_ref(L.lpf, sr);

        const float* __restrict__ S = a.state + vi;
        F.ph = __float_as_uint(S[S_HAS_PHASE * vp]) != 0u ? S[S_PHASE * vp] : 0.0f;   // process.rs:316
        n = __float_as_uint(S[S_OFFSET * vp]);
        if (FILTER == 0) {
            F.fs.y1 = S[S_LAST * vp];
        } else {
            F.fs.x1 = S[S_X1 * vp]; F.fs.x2 = S[S_X2 * vp];
            F.fs.y1 = S[S_Y1 * vp]; F.fs.y2 = S[S_Y2 * vp];
        }
        F.gain = L.gain;
        F.namt = L.namt;
        // memoised derived constants (keys = exact input bits; kNoKey -> first use derives them)
        OscC oc;
        oc.fo_bits = __float_as_uint(S[S_FO_KEY * vp]);
        oc.P = S[S_OSC_P * vp]; oc.d = S[S_OSC_D * vp]; oc.slope = S[S_OSC_SLOPE * vp];
        oc.half = S[S_OSC_HALF * vp]; oc.ts1 = S[S_OSC_TS1 * vp]; oc.ts2 = S[S_OSC_TS2 * vp];
        C.oc = oc;
        FiltC fc;
        fc.fl_bits = __float_as_uint(S[S_DAMP_KEY * vp]) == __float_as_uint(L.damp) ? __float_as_uint(S[S_FL_KEY * vp]) : kNoKey;
        fc.c0 = S[S_FC_C0 * vp]; fc.c1 = S[S_FC_C1 * vp]; fc.c2 = S[S_FC_C2 * vp];
        C.fc = fc;
        C.n_safe = 0u;
        C.msg.es = C.msg.nex0 = C.msg.ey0 = 0.0f; C.msg.nbeg = 1u; C.msg.nend = 0u; C.msg.stage = 4;
        F.seg_end = active ? 0u : 0xffffffffu;
    }
    bool lane_gconst = true;          // the lane's current amp segment (F.es ..) is a sustain / end stage

    // Warp-uniform oscillator kind -> straight-line specialised loop; mixed warps use the per-voice select.
    const uint32_t amask = __ballot_sync(0xffffffffu, active);
    const int leader = amask ? __ffs(amask) - 1 : 0;
    int wkind = -1;
    {
        const uint32_t k0 = __shfl_sync(0xffffffffu, kind, leader);
        if (__all_sync(0xffffffffu, !active || kind == k0)) wkind = (int)k0;
    }
    // +0.0 noise amounts only, and offsets / rotated seeds that are multiples of the trip length; offsets advance by
    // whole 32-frame chunks while on the fast path, so this holds for the launch
    const bool fasthash = __all_sync(0xffffffffu, !active || (__float_as_uint(F.namt) == 0u &&
                                                              ((n | rot) & (uint32_t)(S2_TRIP - 1)) == 0u));

    // Do the active voices of the warp share one cutoff trajectory (cutoff, damping, modulation amount, mod
    // envelope, frame offset)?  Then a moving-cutoff chunk computes its 32 frames' coefficients once, one frame
    // per lane (modcut_coefficients).  Offsets advance together, so this holds for the launch.
    bool filt_uniform = false;
    {
        const EnvQ& M = C.mod;
        const float key[10] = {C.lpf, C.damp, C.amt_lpf, M.A, M.AD, M.S, M.Rs, M.E, M.sD, M.sR};
        // (every lane must execute every shuffle: no short-circuit between them)
        const uint32_t n_lead = __shfl_sync(0xffffffffu, n, leader);
        const float sa_lead = __shfl_sync(0xffffffffu, M.sA, leader);
        bool same = n_lead == n;
        same &= __float_as_uint(sa_lead) == __float_as_uint(M.sA);
#pragma unroll
        for (int k = 0; k < 10; k++)
            same &= __float_as_uint(__shfl_sync(0xffffffffu, key[k], leader)) == __float_as_uint(key[k]);
        filt_uniform = amask != 0u && __all_sync(0xffffffffu, same || !active);
    }

    const uint32_t frames = a.frames;
    const uint32_t f16 = frames & ~15u;            // x16 region (process.rs:26-37), then the scalar tail
    const size_t stride = a.row_stride;
    float* __restrict__ gout = a.voice_out;
    // Output rows are indexed by the caller's voice index, which the bank has permuted (P_ROW).  Transposed
    // write-back of a 64-frame tile: lanes 16q .. 16q+15 cover 256 contiguous bytes of tile row 2*i + q, so each
    // STG.128 of the warp writes two runs of 256 bytes.
    const int q = lane >> 4, c4 = (lane & 15) * 4;
    // rp[tile row] = base address of that voice's output row (0 = none): 32 64-bit words per warp.  The two
    // q-groups of a store read two neighbouring words (broadcast inside a group): conflict-free LDS.64.
    unsigned long long* rp = reinterpret_cast<unsigned long long*>(cold_base + kRows * kColdWords);
    float* ctab = cold_base + kRows * kColdWords + kRows * kRowPtrWords;
    bool all_rows;
    {
        const uint32_t r = C.out_row;
        rp[lane] = (gout && r != 0xffffffffu) ? reinterpret_cast<unsigned long long>(gout + (size_t)r * stride) : 0ull;
        __syncwarp();
        all_rows = __all_sync(0xffffffffu, gout != nullptr && r != 0xffffffffu);   // every tile row has an output row
    }

    // fast_left: frames for which every voice of the warp keeps its resting period and cutoff (warp-uniform);
    // seg_left: frames for which every voice stays inside its current amp-envelope segment, all_gconst: and all of
    // those are sustain / end stages; semi_left: frames for which the moving-cutoff classification holds.
    // 0 = look again before the next chunk.
    uint32_t fast_left = 0, seg_left = 0, semi_left = 0;
    bool all_gconst = false;

    // Runs of tiles.  A third of the warp's stall time sits at the tile boundaries (loop control, dispatch,
    // store-variant selection: uniform-datapath code with exposed latencies, and the warps of an SM reach it in
    // lockstep), so when the store has its simple launch-uniform form — every tile row has an output row or no
    // rows are wanted, and the mix, if any, is the per-warp partial of a wide bank — the fast path renders up to
    // kRunTiles tiles per trip round the outer loop, each followed by its own straight-line write-back.
#ifndef S2_RUN_TILES
#define S2_RUN_TILES 4
#endif
    constexpr uint32_t kRunTiles = S2_RUN_TILES;
    constexpr uint32_t kTile = kTileFrames;
    // this warp's partial row of the mix, from launch parameters and the block index only (uniform registers: a
    // pointer kept live across the chunk loop is spilled under the register cap and reloaded from local memory)
    auto bus_row = [&]() -> float* {
        return a.bus_partials + (size_t)(a.slot_begin / (uint32_t)kRows + blockIdx.x) * a.frames;
    };
    // (16-byte stores into the partial row: needs frames % 4 == 0 and an aligned base)
    const bool bus_wide_ok = a.bus_partials != nullptr && a.n_voices > 32u && (frames & 3u) == 0u &&
                             (reinterpret_cast<uintptr_t>(a.bus_partials) & 15u) == 0u;
    bool simple_store = (gout == nullptr || all_rows) && (a.bus_partials == nullptr || bus_wide_ok);
    if constexpr (!kMeter) simple_store = simple_store && (gout != nullptr || a.bus_partials != nullptr);
    // (a metered launch without rows or a bus stores nothing per tile and takes the runs too)
    // Write-back of a full tile at frame ts.  ROWS: every tile row has an output row; MIX: per-warp partial sums of
    // a wide bank — each lane adds its 16 rows as two pairwise trees of packed adds, then the two q-groups are added
    // by one butterfly shuffle (a fixed tree: deterministic).  `checked`: rows may be missing (rp == 0).
    auto store_tile = [&](uint32_t ts, bool rows, bool mix, bool checked) {
        const size_t tb = ((size_t)ts + (size_t)c4) * sizeof(float);
        if (!mix) {
#pragma unroll
            for (int i = 0; i < 16; i++) {
                char* dst = reinterpret_cast<char*>(rp[2 * i + q]);
                const float4 val = *reinterpret_cast<const float4*>(tile + (2 * i + q) * kTileStride + c4);
                if (!checked || dst) __stcs(reinterpret_cast<float4*>(dst + tb), val);
            }
        } else {
            float2 s01 = make_float2(0.0f, 0.0f), s23 = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
                float4 val[8];
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const int r = 2 * (8 * hh + i) + q;
                    val[i] = *reinterpret_cast<const float4*>(tile + r * kTileStride + c4);
                    if (rows) {
                        char* dst = reinterpret_cast<char*>(rp[r]);
                        if (!checked || dst) __stcs(reinterpret_cast<float4*>(dst + tb), val[i]);
                    }
                }
                float2 t01, t23;
                tree_sum_rows<8>(val, t01, t23);
                s01 = hh ? padd2(s01, t01) : t01;
                s23 = hh ? padd2(s23, t23) : t23;
            }
            s01 = padd2(s01, make_float2(__shfl_xor_sync(0xffffffffu, s01.x, 16), __shfl_xor_sync(0xffffffffu, s01.y, 16)));
            s23 = padd2(s23, make_float2(__shfl_xor_sync(0xffffffffu, s23.x, 16), __shfl_xor_sync(0xffffffffu, s23.y, 16)));
            if (lane < 16) *reinterpret_cast<float4*>(bus_row() + ts + c4) = make_float4(s01.x, s01.y, s23.x, s23.y);
        }
    };
    // The amp envelope of the lanes whose segment ends inside a chunk that ran with a gain of exactly 1 (the packed
    // loops take the envelope as one line): out = RN(y * g), as every other path rounds it.  The warp does one such
    // lane at a time, one frame per lane, from that lane's envelope in shared memory.  `h` = the chunk's first
    // column of the tile, `n0` = each lane's own frame offset at the chunk's start.
    auto edge_gain = [&](bool edge, uint32_t h, uint32_t n0) {
        uint32_t em = __ballot_sync(0xffffffffu, edge);
        if (em == 0u) return;
        __syncwarp();
        while (em) {
            const int l = __ffs(em) - 1;
            em &= em - 1u;
            const Cold& CL = *reinterpret_cast<const Cold*>(cold_base + l * kColdWords);
            const uint32_t nl = __shfl_sync(0xffffffffu, n0, l);
            float* r = tile + l * kTileStride + h + lane;
            *r = __fmul_rn(*r, env_x16(CL.amp, __uint2float_rn(nl + (uint32_t)lane)));
        }
        __syncwarp();
    };
    auto clear_chunk = [&](float* r) {
#pragma unroll
        for (int j = 0; j < kChunk / 4; j++)
            *reinterpret_cast<float4*>(r + 4 * j) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    };

    for (uint32_t t0 = 0; t0 < frames; t0 += kTile) {
        const uint32_t tcnt = min(kTile, frames - t0);
        bool written = false;              // a run of fast tiles writes its tiles back itself
        for (uint32_t h0 = 0; h0 < tcnt; h0 += kChunk) {
            const uint32_t tc = t0 + h0;               // first frame of this chunk
            float* crow = row + h0;
            const uint32_t cnt = min((uint32_t)kChunk, frames - tc);
            const bool full = cnt == kChunk && tc + kChunk <= f16 && a.force_path != 2u;
            bool warp_fast = full && fast_left >= (uint32_t)kChunk;
            bool warp_semi = full && !warp_fast && semi_left >= (uint32_t)kChunk;
            if (full && !warp_fast && !warp_semi) {
                // (Re)classify: which envelope segments is frame n in, and until when.
                bool lane_fast = !active, lane_semi = !active;
                uint32_t lane_left = 0xffffffffu;          // frames this lane's classification holds for
                if (active) {
                    lane_fast = n + kChunk <= C.n_safe;
                    if (!lane_fast) {
                        const bool mm = (C.flags & 2u) != 0u;
                        SegEnv sm = {0.0f, 0.0f, 0.0f, 0u, 1u << 24, 4};
                        if (mm && n < (1u << 24)) sm = seg_env(C.mod, n);
                        const bool mconst = !mm || !stage_moves(sm.stage);
                        uint32_t n_safe = 0u;
                        if (mconst && n < (1u << 24)) {
                            // resting: the mod envelope is constant (sustain / end) or nothing follows it
                            n_safe = mm ? sm.nend : 1u << 24;
                            const float m = (mm && sm.stage == 2) ? C.mod.S : 0.0f;
                            const float fo = modulate_freq(C.pitch, m, C.amt_osc);
                            const float fl = modulate_freq(C.lpf, m, C.amt_lpf);
                            OscC oc = C.oc;
                            FiltC fc = C.fc;
                            if (__float_as_uint(fo) != oc.fo_bits) { make_osc(oc, fo, sr); C.oc = oc; }
                            if (__float_as_uint(fl) != fc.fl_bits) { make_filt<FILTER>(fc, fl, C.damp, sr); C.fc = fc; }
                            // the fast phase step needs 1/P < 1 (and a sane period)
                            const bool sane = oc.d < 1.0f && oc.P > 1.0f;
                            if (!sane) n_safe = 0u;
                            lane_fast = sane && n + kChunk <= n_safe;
                            // publish into the lane's registers
                            set_osc(F, oc);
                            F.fc = fc;
                        } else if (!mconst && C.amt_osc == 0.0f && n + kChunk <= sm.nend) {
                            // the mod envelope ramps through the whole chunk and only the cutoff follows it: the period
                            // is the per-voice constant sr / pitch -> moving-cutoff chunk
                            OscC oc = C.oc;
                            if (__float_as_uint(C.pitch) != oc.fo_bits) { make_osc(oc, C.pitch, sr); C.oc = oc; }
                            if (oc.d < 1.0f && oc.P > 1.0f) {
                                lane_semi = true;
                                C.msg = sm;
                                set_osc(F, oc);
                            }
                        }
                        C.n_safe = n_safe;
                    }
                    if (lane_fast) { lane_left = C.n_safe - n; C.flags &= ~4u; }
                    else if (lane_semi) { lane_left = C.msg.nend - n; C.flags |= 4u; }
                    lane_semi |= lane_fast;
                }
                warp_fast = amask != 0u && __all_sync(0xffffffffu, lane_fast);
                warp_semi = !warp_fast && amask != 0u && __all_sync(0xffffffffu, lane_semi);
                fast_left = semi_left = 0;
                if (warp_fast) fast_left = __reduce_min_sync(0xffffffffu, lane_left);
                if (warp_semi) semi_left = __reduce_min_sync(0xffffffffu, lane_left);
            }

            if (warp_fast) {
                if (seg_left < (uint32_t)kChunk) {
                    // some lane's amp-envelope segment ends inside this chunk, or is not known yet: look again
                    if (active && n >= F.seg_end) {
                        const SegEnv sg = seg_env(C.amp, n);
                        F.es = sg.es; F.nex0 = sg.nex0; F.ey0 = sg.ey0; F.seg_end = sg.nend;
                        lane_gconst = sg.stage == 2 || sg.stage == 4;
                    }
                    seg_left = __reduce_min_sync(0xffffffffu, active ? F.seg_end - n : 0xffffffffu);
                    all_gconst = __all_sync(0xffffffffu, lane_gconst);
                }
                // A stage boundary of some lane's amp envelope inside the chunk (banks of the fast hash form): those
                // lanes run the chunk with a gain of exactly 1 and multiply their 32 frames by the envelope
                // afterwards (edge_gain) — one rounding either way.
                bool edge = false;
                int gmode = all_gconst ? G_CONST : G_LINE;
                if (seg_left < (uint32_t)kChunk) {
                    gmode = G_ANY;
                    if (fasthash) {
                        gmode = G_LINE;
                        edge = active && F.seg_end - n < (uint32_t)kChunk;
                        if (edge) { F.es = 0.0f; F.nex0 = 0.0f; F.ey0 = 1.0f; }
                    }
                }
                // Run: whole tiles for as long as the classification holds, each with its straight-line write-back
                // (inactive voices run the same code on zeroed constants; their rows are cleared)
                uint32_t reps = 0;
                if (simple_store && seg_left >= kTile && h0 == 0u && tcnt == kTile)
                    reps = min(min(min(fast_left, seg_left), f16 - t0) / kTile, kRunTiles);
                const uint32_t n_chunks = reps ? reps * (kTile / (uint32_t)kChunk) : 1u;
                uint32_t hh = h0, ts = t0;
                for (uint32_t k = 0; k < n_chunks; k++) {
                    with_kind<0, 1, 2, 3, -1>(wkind, [](auto K, auto&&... args) { fast_tile<FILTER, K, TRACE>(args...); },
                                              gmode, fasthash, F, &C.amp, one, kind, rot, n, row + hh, sintab);
                    if (TRACE != TRACE_PHASE && seg_left < (uint32_t)kChunk) edge_gain(edge, hh, n);
                    n += kChunk;
                    hh += (uint32_t)kChunk;
                    if (reps && hh == kTile) {
                        if (!active) { clear_chunk(row); clear_chunk(row + kChunk); }
                        __syncwarp();
                        if constexpr (kMeter) {
                            // the lane's own row of the finished tile into its meters (inactive lanes reduce their
                            // cleared rows: no divergence)
                            if (gout != nullptr || a.bus_partials != nullptr)
                                store_tile(ts, gout != nullptr, a.bus_partials != nullptr, false);
                            meter_row(row, kTile, one, meter_sum(smem)[lane], meter_peak(smem)[lane]);
                        } else {
                            store_tile(ts, gout != nullptr, a.bus_partials != nullptr, false);
                        }
                        __syncwarp();      // every lane is done reading the tile before the next one overwrites it
                        hh = 0u;
                        ts += kTile;
                    }
                }
                fast_left -= n_chunks * (uint32_t)kChunk;
                seg_left = seg_left < (uint32_t)kChunk ? 0u : seg_left - n_chunks * (uint32_t)kChunk;
                if (reps) {
                    t0 += (reps - 1u) * kTile;               // the loop header adds the last tile
                    written = true;
                    break;
                }
            } else if (warp_semi) {
                // Moving-cutoff chunk.  Lanes whose cutoff rests (flag 4 clear) run the same code on their constants.
                MovV mv;
                mv.moving = active && (C.flags & 4u) != 0u;
                mv.cp = cutp_of(C.lpf, C.theta0, C.amt_lpf, C.damp, sr, rsr);
                SegEnv sm = C.msg;
                mv.mes = sm.es; mv.mnex0 = sm.nex0; mv.mey0 = sm.ey0;
                constexpr bool kPackable = FILTER == FILT_ONE_POLE || FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP;
                constexpr bool kPairable = FILTER == FILT_BIQUAD_LP || FILTER == FILT_BIQUAD_HP;
                // the packed forms take the amp envelope as one line through the chunk (as G_LINE); a lane with a stage
                // boundary inside the chunk takes a gain of 1 and edge_gain afterwards
                auto amp_line = [&]() {
                    if (active && n >= F.seg_end) {
                        const SegEnv sg = seg_env(C.amp, n);
                        F.es = sg.es; F.nex0 = sg.nex0; F.ey0 = sg.ey0; F.seg_end = sg.nend;
                        lane_gconst = sg.stage == 2 || sg.stage == 4;
                    }
                    const bool edge = active && F.seg_end - n < (uint32_t)kChunk;
                    if (edge) { F.es = 0.0f; F.nex0 = 0.0f; F.ey0 = 1.0f; }
                    return edge;
                };
                const bool packable = a.force_path == 0u || a.force_path == 3u;
                if (filt_uniform) {
                    // one cutoff trajectory for the whole warp: 32 frames' coefficients, one per lane, once; the
                    // chunk reads them
                    const Cold& CL = *reinterpret_cast<const Cold*>(cold_base + leader * kColdWords);
                    const uint32_t n_lead = __shfl_sync(0xffffffffu, n, leader);   // inactive lanes hold other offsets
                    const CutP cpl = cutp_of(CL.lpf, CL.theta0, CL.amt_lpf, CL.damp, sr, rsr);
                    const SegEnv sml = CL.msg;
                    modcut_coefficients<FILTER>(sml, cpl, one, n_lead, lane, ctab);
                    __syncwarp();
                    if (packable) {
                        const bool edge = amp_line();
                        s2c::Window W;
                        window_none(W);
                        with_kind<0, 1, -1>(wkind, [](auto K, auto&&... args) { chunk_modcut_pk<FILTER, K, TRACE, true>(args...); },
                                            F, mv, W, one, kind, rot, n, crow, sintab, ctab);
                        if (TRACE != TRACE_PHASE) edge_gain(edge, h0, n);
                    } else {
                        chunk_modcut_sc<FILTER, -1, TRACE, true>(F, &C.amp, mv, sm, one, kind, rot, n, crow, sintab, ctab);
                    }
                    __syncwarp();          // ctab is rewritten by the next moving-cutoff chunk
                } else {
                    // each lane's own coefficients: packed where every moving lane is aligned and (second-order filters)
                    // has a valid window, paired where moreover no lane pair (2i, 2i + 1) holds two moving lanes (the
                    // resting lane of a pair helps); otherwise one frame at a time
                    enum { ONE_FRAME, PACKED, PAIRED };
                    int form = ONE_FRAME;
                    bool edge = false;
                    s2c::Window W;
                    window_none(W);
                    if constexpr (kPackable) {
                        edge = amp_line();
                        bool ok = true;
                        if (mv.moving) {
                            ok = (n & 31u) == 0u;
                            if (FILTER != FILT_ONE_POLE && ok) {
                                make_window_inl<FILTER>(W, sm, mv.cp, n);
                                ok = W.valid != 0u;
                            }
                        }
                        if (packable && __all_sync(0xffffffffu, ok)) {
                            const uint32_t mmask = __ballot_sync(0xffffffffu, mv.moving);
                            form = kPairable && (mmask & (mmask >> 1) & 0x55555555u) == 0u && a.force_path != 3u ? PAIRED : PACKED;
                        }
                    }
                    if (form == PAIRED) {
                        if constexpr (kPairable)
                            with_kind<0, 1, -1>(wkind, [](auto K, auto&&... args) { chunk_modcut_pr<FILTER, K, TRACE>(args...); },
                                                F, mv, W, one, kind, rot, n, crow, sintab);
                    } else if (form == PACKED) {
                        if constexpr (kPackable)
                            with_kind<0, 1, -1>(wkind, [](auto K, auto&&... args) { chunk_modcut_pk<FILTER, K, TRACE>(args...); },
                                                F, mv, W, one, kind, rot, n, crow, sintab);
                    } else {
                        chunk_modcut_sc<FILTER, -1, TRACE, false>(F, &C.amp, mv, sm, one, kind, rot, n, crow, sintab, nullptr);
                    }
                    if (TRACE != TRACE_PHASE && form != ONE_FRAME) edge_gain(edge, h0, n);
                }
                n += kChunk;
                semi_left -= (uint32_t)kChunk;
                seg_left = 0u;             // the amp segment registers were not kept up to date
            } else {
                if (active) {
                    // the general path derives everything again from the voice's parameter column
                    const Lane L = load_lane(a.params + C.vi, vp, sr, C.release);
                    OscC oc = C.oc;
                    FiltC fc = C.fc;
                    MovG mg;
                    movg_init(mg, L.lpf, L.amt_lpf, L.damp, sr);
                    for (uint32_t i = 0; i < cnt; i++) {
                        const bool scalar_sem = tc + i >= f16;
                        crow[i] = general_frame<FILTER, TRACE>(L, sr, one, n, scalar_sem, oc, fc, mg, F.ph, F.fs, sintab);
                        n += 1u;
                    }
                    C.oc = oc;
                    C.fc = fc;
                    C.n_safe = 0u;         // oc/fc may have moved: republish through the classifier
                }
                fast_left = semi_left = seg_left = 0u;
            }
            if (!active) clear_chunk(crow);
        }
        if (written) continue;
        // ---- write-back of this tile (tcnt frames)
        __syncwarp();
        float* __restrict__ gbus = a.bus_partials ? bus_row() : nullptr;
        const bool wide_bus = gbus != nullptr && bus_wide_ok && tcnt == kTile;
        if (tcnt == kTile && (gout || wide_bus)) {
            store_tile(t0, gout != nullptr, wide_bus, !all_rows);
        } else if (gout) {
            for (uint32_t r = 0; r < 32u; r++) {
                const uint32_t orow = __shfl_sync(0xffffffffu, C.out_row, r);
                if (orow != 0xffffffffu)
                    for (uint32_t c = (uint32_t)lane; c < tcnt; c += 32u)
                        gout[(size_t)orow * stride + t0 + c] = tile[r * kTileStride + c];
            }
        }
        if (gbus && !wide_bus) {
            for (uint32_t c = (uint32_t)lane; c < tcnt; c += 32u) {
                float acc;
                if (a.n_voices <= 32u) {
                    // synth.rs:176-202: voices are accumulated in index order, starting from 0.0 — the
                    // reference's exact summation order (a bank this narrow is one warp, identity slots)
                    acc = 0.0f;
#pragma unroll 8
                    for (int r = 0; r < kRows; r++) acc = __fadd_rn(acc, tile[r * kTileStride + c]);
                } else {
                    // ragged last tile of a wide bank: fixed 4-way tree over the warp's rows
                    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
                    for (int r = 0; r < kRows; r += 4) {
                        a0 = __fadd_rn(a0, tile[(r + 0) * kTileStride + c]);
                        a1 = __fadd_rn(a1, tile[(r + 1) * kTileStride + c]);
                        a2 = __fadd_rn(a2, tile[(r + 2) * kTileStride + c]);
                        a3 = __fadd_rn(a3, tile[(r + 3) * kTileStride + c]);
                    }
                    acc = __fadd_rn(__fadd_rn(a0, a1), __fadd_rn(a2, a3));
                }
                gbus[t0 + c] = acc;
            }
        }
        if constexpr (kMeter) meter_row(row, tcnt, one, meter_sum(smem)[lane], meter_peak(smem)[lane]);
        __syncwarp();      // every lane is done reading the tile before the next one overwrites it
    }

    if (active) {
        float* __restrict__ S = a.state + C.vi;
        S[S_PHASE * vp] = F.ph;
        S[S_HAS_PHASE * vp] = __uint_as_float(1u);
        const uint32_t start = __float_as_uint(S[S_OFFSET * vp]);
        const uint32_t nxt = start + frames < start ? 0xffffffffu : start + frames;   // saturating (synth.rs:197)
        S[S_OFFSET * vp] = __uint_as_float(nxt);
        if (FILTER == 0) S[S_LAST * vp] = F.fs.y1;
        else {
            S[S_X1 * vp] = F.fs.x1; S[S_X2 * vp] = F.fs.x2;
            S[S_Y1 * vp] = F.fs.y1; S[S_Y2 * vp] = F.fs.y2;
        }
        const OscC oc = C.oc;
        const FiltC fc = C.fc;
        S[S_FO_KEY * vp] = __uint_as_float(oc.fo_bits);
        S[S_OSC_P * vp] = oc.P; S[S_OSC_D * vp] = oc.d; S[S_OSC_SLOPE * vp] = oc.slope;
        S[S_OSC_HALF * vp] = oc.half; S[S_OSC_TS1 * vp] = oc.ts1; S[S_OSC_TS2 * vp] = oc.ts2;
        S[S_FL_KEY * vp] = __uint_as_float(fc.fl_bits);
        S[S_DAMP_KEY * vp] = C.damp;
        S[S_FC_C0 * vp] = fc.c0; S[S_FC_C1 * vp] = fc.c1; S[S_FC_C2 * vp] = fc.c2;
        if constexpr (kMeter) {
            // a voice is one lane of one launch, and a voice range's launches are stream-ordered: no atomics
            const uint32_t r = C.out_row;
            a.sum_sq[r] = __dadd_rn(a.sum_sq[r], meter_sum(smem)[lane]);
            a.peak[r] = max(a.peak[r], meter_peak(smem)[lane]);
        }
    }
}

// Bus reduction: one kernel, fixed summation order (deterministic).  Block fx owns 32 frames; its 8 warps take the
// partial rows w, w + 8, w + 16, ... (lane = frame: 128-byte coalesced reads), each with four accumulators over
// consecutive rows of its sequence, eight loads in flight; the eight warp sums are then added in order.
// Few, long-lived blocks on purpose: the reduction runs next to the render kernels of the following step on a
// machine whose every slot is taken by long-running render blocks.  The 4,096 short blocks of the two-stage
// form it replaces queued for those slots one by one and cost ~30 us of step time for 19 us of work; 128 blocks
// of 8 warps need one slot each and displace next to nothing (it is latency-bound at ~20 us, off the critical path).
__global__ void __launch_bounds__(256) bus_reduce_kernel(const float* __restrict__ partials, uint32_t n_rows,
                                                         size_t row_stride, uint32_t frames, float* __restrict__ bus) {
    __shared__ float sm[8][33];
    const uint32_t tx = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t t = blockIdx.x * 32u + tx;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    if (t < frames) {
        const float* __restrict__ col = partials + t;
        uint32_t r = w;
        for (; r + 56u < n_rows; r += 64u) {                  // rows r, r+8, ..., r+56: eight loads in flight
            float v[8];
#pragma unroll
            for (uint32_t k = 0; k < 8u; k++) v[k] = col[(size_t)(r + 8u * k) * row_stride];
            a0 = __fadd_rn(a0, v[0]); a1 = __fadd_rn(a1, v[1]); a2 = __fadd_rn(a2, v[2]); a3 = __fadd_rn(a3, v[3]);
            a0 = __fadd_rn(a0, v[4]); a1 = __fadd_rn(a1, v[5]); a2 = __fadd_rn(a2, v[6]); a3 = __fadd_rn(a3, v[7]);
        }
        for (uint32_t k = 0; r < n_rows; r += 8u, k++) {     // the rest, same rotation over the accumulators
            const float v = col[(size_t)r * row_stride];
            if ((k & 3u) == 0u) a0 = __fadd_rn(a0, v);
            else if ((k & 3u) == 1u) a1 = __fadd_rn(a1, v);
            else if ((k & 3u) == 2u) a2 = __fadd_rn(a2, v);
            else a3 = __fadd_rn(a3, v);
        }
    }
    sm[w][tx] = __fadd_rn(__fadd_rn(a0, a1), __fadd_rn(a2, a3));
    __syncthreads();
    if (w == 0 && t < frames) {
        float total = sm[0][tx];
#pragma unroll
        for (int k = 1; k < 8; k++) total = __fadd_rn(total, sm[k][tx]);
        bus[t] = total;
    }
}

// The same reduction for wide banks, four frames per lane: block (fx, rs) owns 128 frames and a quarter of the
// partial rows; its 8 warps take the rows w, w + 8, ... of that quarter with 16-byte loads (512 contiguous bytes per
// warp and row, four rows in flight per lane: four times the bytes in flight of the form above, a quarter of its
// instructions), the quarter's sum goes to `scratch[rs]`, and the last of the four blocks to finish adds the four
// quarters in index order — a fixed order whichever block that is.  It shares the machine with the render blocks of
// the next step for a third of the time the one-frame-per-lane form needs.
constexpr uint32_t kRedSplit = 4;

__global__ void __launch_bounds__(256, 8) bus_reduce_wide_kernel(const float* __restrict__ partials, uint32_t n_rows,
                                                              size_t row_stride, uint32_t frames, float* scratch,
                                                              unsigned int* counters, float* __restrict__ bus) {
    __shared__ float4 sm[8][32];
    __shared__ bool last;
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t fx = blockIdx.x / kRedSplit, rs = blockIdx.x % kRedSplit;
    const uint32_t t = fx * 128u + 4u * lane;
    const uint32_t r1 = (uint32_t)((uint64_t)n_rows * (rs + 1u) / kRedSplit);
    uint32_t r = (uint32_t)((uint64_t)n_rows * rs / kRedSplit) + w;
    auto add4 = [](float4 a, float4 v) {
        return make_float4(__fadd_rn(a.x, v.x), __fadd_rn(a.y, v.y), __fadd_rn(a.z, v.z), __fadd_rn(a.w, v.w));
    };
    float4 a0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), a1 = a0;
    const float* __restrict__ col = partials + t;
    for (; r + 24u < r1; r += 32u) {                        // rows r, r + 8, r + 16, r + 24 in flight
        float4 v[4];
#pragma unroll
        for (uint32_t k = 0; k < 4u; k++) v[k] = __ldcs(reinterpret_cast<const float4*>(col + (size_t)(r + 8u * k) * row_stride));
        a0 = add4(a0, v[0]); a1 = add4(a1, v[1]); a0 = add4(a0, v[2]); a1 = add4(a1, v[3]);
    }
    for (uint32_t k = 0; r < r1; r += 8u, k++) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(col + (size_t)r * row_stride));
        if (k & 1u) a1 = add4(a1, v); else a0 = add4(a0, v);
    }
    sm[w][lane] = add4(a0, a1);
    __syncthreads();
    if (w == 0) {
        float4 total = sm[0][lane];
#pragma unroll
        for (int k = 1; k < 8; k++) total = add4(total, sm[k][lane]);
        __stcg(reinterpret_cast<float4*>(scratch + (size_t)rs * frames + t), total);
        __threadfence();
    }
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&counters[fx], 1u) == kRedSplit - 1u;
    __syncthreads();
    if (last && w == 0) {
        __threadfence();
        float4 total = __ldcg(reinterpret_cast<const float4*>(scratch + t));
#pragma unroll
        for (uint32_t k = 1; k < kRedSplit; k++) total = add4(total, __ldcg(reinterpret_cast<const float4*>(scratch + (size_t)k * frames + t)));
        *reinterpret_cast<float4*>(bus + t) = total;
        if (lane == 0) counters[fx] = 0u;                  // ready for the next launch (same stream)
    }
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ staged, const float* __restrict__ row_index_bits,
                                  uint32_t* __restrict__ dst, uint32_t n) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) dst[s] = staged[__float_as_uint(row_index_bits[s])];
}

cudaError_t launch_gather_u32(const uint32_t* staged, const float* row_index_bits, uint32_t* dst_row,
                              uint32_t n, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    gather_u32_kernel<<<(n + 255) / 256, 256, 0, stream>>>(staged, row_index_bits, dst_row, n);
    return cudaGetLastError();
}

// Bulk note-on: thread j takes entry e = begin + j of the packed batch (one column per entry, read coalesced across
// the entries) and writes its P_COUNT + S_COUNT words at its slot.  A pending note-off table gets the entry's release
// offset at the entry's voice index, so that the render prologue that applies the table keeps the note-on's value.
__global__ void set_voices_kernel(const float* __restrict__ batch, uint32_t m, uint32_t begin, uint32_t count,
                                  float* __restrict__ params, float* __restrict__ state, uint32_t vpad,
                                  uint32_t* __restrict__ staged_release) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= count) return;
    const size_t e = begin + j;
    const size_t slot = __float_as_uint(batch[(size_t)(P_COUNT + S_COUNT) * m + e]);
#pragma unroll
    for (int k = 0; k < P_COUNT; k++) params[(size_t)k * vpad + slot] = batch[(size_t)k * m + e];
#pragma unroll
    for (int k = 0; k < S_COUNT; k++) state[(size_t)k * vpad + slot] = batch[(size_t)(P_COUNT + k) * m + e];
    if (staged_release != nullptr)
        staged_release[__float_as_uint(batch[(size_t)P_ROW * m + e])] = __float_as_uint(batch[(size_t)P_RELEASE * m + e]);
}

cudaError_t launch_set_voices(const float* batch, uint32_t m, uint32_t begin, uint32_t count, float* params,
                              float* state, uint32_t vpad, uint32_t* staged_release, cudaStream_t stream) {
    if (count == 0) return cudaSuccess;
    set_voices_kernel<<<(count + 255) / 256, 256, 0, stream>>>(batch, m, begin, count, params, state, vpad, staged_release);
    return cudaGetLastError();
}

uint32_t render_warps(uint32_t n_voices) { return (n_voices + 31u) / 32u; }

static_assert((warp_smem_floats() + kMeterFloats) * sizeof(float) + 4096 <= 48 * 1024,
              "the render kernel's dynamic shared memory must stay under the 48 KB that needs no opt-in");
// A bank of 65,536 voices without sine voices needs 13.8 blocks per SM resident at once, metered or not: 14 blocks of
// the metered size plus the 1 KB the runtime reserves per block (128-byte granules) fit the 228 KB of an SM.
static_assert(14 * (((warp_smem_floats() + kMeterFloats) * sizeof(float) + 127) / 128 * 128 + 1024) <= 228 * 1024,
              "a metered launch must keep 14 resident blocks per SM");

// One warp per block (DESIGN.md section 4.2).
template <int FILTER, int TRACE>
static cudaError_t launch_t(const RenderArgs& a, cudaStream_t stream) {
    const size_t smem = (warp_smem_floats() + (TRACE == TRACE_METER ? kMeterFloats : 0)) * sizeof(float) +
                        (a.has_sine ? 4096 : 0);
    render_kernel<FILTER, TRACE><<<render_warps(a.slot_end - a.slot_begin), 32, smem, stream>>>(a);
    return cudaGetLastError();
}

template <int FILTER>
static cudaError_t launch_f(const RenderArgs& a, int trace, cudaStream_t stream) {
    if (trace == TRACE_PHASE) return launch_t<FILTER, TRACE_PHASE>(a, stream);
    return a.sum_sq ? launch_t<FILTER, TRACE_METER>(a, stream) : launch_t<FILTER, TRACE_NONE>(a, stream);
}

cudaError_t launch_render(const RenderArgs& a, uint32_t filter_kind, int trace, cudaStream_t stream) {
    if (a.n_voices == 0 || a.frames == 0) return cudaSuccess;
    switch (filter_kind) {
    case FILT_ONE_POLE: return launch_f<FILT_ONE_POLE>(a, trace, stream);
    case FILT_BIQUAD_LP: return launch_f<FILT_BIQUAD_LP>(a, trace, stream);
    case FILT_BIQUAD_HP: return launch_f<FILT_BIQUAD_HP>(a, trace, stream);
    case FILT_BIQUAD_BP: return launch_f<FILT_BIQUAD_BP>(a, trace, stream);
    case FILT_FIRST_LP: return launch_f<FILT_FIRST_LP>(a, trace, stream);
    case FILT_FIRST_HP: return launch_f<FILT_FIRST_HP>(a, trace, stream);
    default: return cudaErrorInvalidValue;
    }
}

size_t bus_scratch_floats(uint32_t n_rows, uint32_t frames) {
    const bool wide = n_rows >= 512u && (frames & 127u) == 0u && frames / 128u <= kBusCounters;
    return wide ? (size_t)kRedSplit * frames : 0;
}

cudaError_t launch_bus_reduce(const float* partials, uint32_t n_warps, size_t row_stride, uint32_t frames, float* bus,
                              cudaStream_t stream, unsigned int* counters, float* scratch) {
    if (frames == 0) return cudaSuccess;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15u) == 0u; };
    const bool wide = counters != nullptr && scratch != nullptr && bus_scratch_floats(n_warps, frames) != 0 &&
                      (row_stride & 3u) == 0u && al16(partials) && al16(scratch) && al16(bus);
    if (wide)
        bus_reduce_wide_kernel<<<frames / 128u * kRedSplit, 256, 0, stream>>>(partials, n_warps, row_stride, frames, scratch,
                                                                              counters, bus);
    else
        bus_reduce_kernel<<<(frames + 31) / 32, 256, 0, stream>>>(partials, n_warps, row_stride, frames, bus);
    return cudaGetLastError();
}

}  // namespace s2
