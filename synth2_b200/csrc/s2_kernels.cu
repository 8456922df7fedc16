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

// The mixed kernel's warp belongs to a bus of at most 32 voices, so its partial adds in voice order from +0.0 (a
// single-kind bank tests its own width instead; a routed bank's buses have any width).
__device__ __forceinline__ bool narrow_bus(const RenderArgs& a) {
    return (a.warp_kinds[a.slot_begin / 32u + blockIdx.x] & kWarpNarrowBus) != 0u;
}

// 65,536 voices = 13.8 one-warp blocks per SM: without pipelining all of them must be resident at once (a
// second wave would serialise: measured +20 % time at 144 registers, where only 13 fit).
template <int FILTER, int TRACE>
__global__ void __launch_bounds__(32, S2_MINBLOCKS)
render_kernel(const RenderArgs a) {
    constexpr bool MIXED = false;
#include "s2_render_body.inc"
}

// The same body for one warp of a mixed-filter bank.  Included rather than called: as a __forceinline__ function
// shared with render_kernel the body is optimised before it is inlined, without the kernel's one-warp bound, and
// eight of the eighteen render_kernel instantiations then compile to different code.
template <int FILTER, int TRACE>
__device__ __forceinline__ void render_body_mixed(const RenderArgs a) {   // by value: no spills (by reference: 16 B)
    constexpr bool MIXED = true;
#include "s2_render_body.inc"
}

// Mixed-filter banks: every warp is kind-uniform (s2_bank_create_mixed), so each block reads its warp's kind once and
// runs that kind's body.  One launch renders every kind: blocks of all kinds fill the machine together, where one
// launch per kind, in turn on one stream, would leave most of it idle for a kind group's few hundred blocks.
template <int TRACE>
__global__ void __launch_bounds__(32, S2_MINBLOCKS)
render_kernel_mixed(const RenderArgs a) {
    switch (a.warp_kinds[a.slot_begin / 32u + blockIdx.x] & kWarpKindMask) {
    case FILT_ONE_POLE: render_body_mixed<FILT_ONE_POLE, TRACE>(a); break;
    case FILT_BIQUAD_LP: render_body_mixed<FILT_BIQUAD_LP, TRACE>(a); break;
    case FILT_BIQUAD_HP: render_body_mixed<FILT_BIQUAD_HP, TRACE>(a); break;
    case FILT_BIQUAD_BP: render_body_mixed<FILT_BIQUAD_BP, TRACE>(a); break;
    case FILT_FIRST_LP: render_body_mixed<FILT_FIRST_LP, TRACE>(a); break;
    default: render_body_mixed<FILT_FIRST_HP, TRACE>(a); break;
    }
}

// Row accessors of the bus reductions: row r of a standalone bank's partial rows (or voice rows), and row r of one
// bus of a routed bank, found through that bus's list of partial rows (its warps) or voice rows.  The summation trees
// below take either, so a routed bank's bus adds its rows in the order a standalone bank of its voices adds them.
struct StridedRows {
    const float* base;
    size_t stride;
    __device__ __forceinline__ const float* operator()(uint32_t r) const { return base + (size_t)r * stride; }
};
struct ListedRows {
    const float* base;
    size_t stride;
    const uint32_t* idx;
    __device__ __forceinline__ const float* operator()(uint32_t r) const { return base + (size_t)__ldg(idx + r) * stride; }
};

// Bus reduction: one kernel, fixed summation order (deterministic).  Block fx owns 32 frames; its 8 warps take the
// partial rows w, w + 8, w + 16, ... (lane = frame: 128-byte coalesced reads), each with four accumulators over
// consecutive rows of its sequence, eight loads in flight; the eight warp sums are then added in order.
// Few, long-lived blocks on purpose: the reduction runs next to the render kernels of the following step on a
// machine whose every slot is taken by long-running render blocks.  The 4,096 short blocks of the two-stage
// form it replaces queued for those slots one by one and cost ~30 us of step time for 19 us of work; 128 blocks
// of 8 warps need one slot each and displace next to nothing (it is latency-bound at ~20 us, off the critical path).
template <class Rows>
__device__ __forceinline__ void bus_reduce_tree(Rows rows, uint32_t n_rows, uint32_t frames, float* __restrict__ bus,
                                                uint32_t fx) {
    __shared__ float sm[8][33];
    const uint32_t tx = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t t = fx * 32u + tx;
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    if (t < frames) {
        uint32_t r = w;
        for (; r + 56u < n_rows; r += 64u) {                  // rows r, r+8, ..., r+56: eight loads in flight
            float v[8];
#pragma unroll
            for (uint32_t k = 0; k < 8u; k++) v[k] = rows(r + 8u * k)[t];
            a0 = __fadd_rn(a0, v[0]); a1 = __fadd_rn(a1, v[1]); a2 = __fadd_rn(a2, v[2]); a3 = __fadd_rn(a3, v[3]);
            a0 = __fadd_rn(a0, v[4]); a1 = __fadd_rn(a1, v[5]); a2 = __fadd_rn(a2, v[6]); a3 = __fadd_rn(a3, v[7]);
        }
        for (uint32_t k = 0; r < n_rows; r += 8u, k++) {     // the rest, same rotation over the accumulators
            const float v = rows(r)[t];
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

__global__ void __launch_bounds__(256) bus_reduce_kernel(const float* __restrict__ partials, uint32_t n_rows,
                                                         size_t row_stride, uint32_t frames, float* __restrict__ bus) {
    bus_reduce_tree(StridedRows{partials, row_stride}, n_rows, frames, bus, blockIdx.x);
}

// The same reduction for wide banks, four frames per lane: block (fx, rs) owns 128 frames and a quarter of the
// partial rows; its 8 warps take the rows w, w + 8, ... of that quarter with 16-byte loads (512 contiguous bytes per
// warp and row, four rows in flight per lane: four times the bytes in flight of the form above, a quarter of its
// instructions), the quarter's sum goes to `scratch[rs]`, and the last of the four blocks to finish adds the four
// quarters in index order — a fixed order whichever block that is.  It shares the machine with the render blocks of
// the next step for a third of the time the one-frame-per-lane form needs.
constexpr uint32_t kRedSplit = 4;

template <class Rows>
__device__ __forceinline__ void bus_reduce_wide_tree(Rows rows, uint32_t n_rows, uint32_t frames, float* scratch,
                                                     unsigned int* counters, float* __restrict__ bus, uint32_t block) {
    __shared__ float4 sm[8][32];
    __shared__ bool last;
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    const uint32_t fx = block / kRedSplit, rs = block % kRedSplit;
    const uint32_t t = fx * 128u + 4u * lane;
    const uint32_t r1 = (uint32_t)((uint64_t)n_rows * (rs + 1u) / kRedSplit);
    uint32_t r = (uint32_t)((uint64_t)n_rows * rs / kRedSplit) + w;
    auto add4 = [](float4 a, float4 v) {
        return make_float4(__fadd_rn(a.x, v.x), __fadd_rn(a.y, v.y), __fadd_rn(a.z, v.z), __fadd_rn(a.w, v.w));
    };
    float4 a0 = make_float4(0.0f, 0.0f, 0.0f, 0.0f), a1 = a0;
    for (; r + 24u < r1; r += 32u) {                        // rows r, r + 8, r + 16, r + 24 in flight
        float4 v[4];
#pragma unroll
        for (uint32_t k = 0; k < 4u; k++) v[k] = __ldcs(reinterpret_cast<const float4*>(rows(r + 8u * k) + t));
        a0 = add4(a0, v[0]); a1 = add4(a1, v[1]); a0 = add4(a0, v[2]); a1 = add4(a1, v[3]);
    }
    for (uint32_t k = 0; r < r1; r += 8u, k++) {
        const float4 v = __ldcs(reinterpret_cast<const float4*>(rows(r) + t));
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

__global__ void __launch_bounds__(256, 8) bus_reduce_wide_kernel(const float* __restrict__ partials, uint32_t n_rows,
                                                              size_t row_stride, uint32_t frames, float* scratch,
                                                              unsigned int* counters, float* __restrict__ bus) {
    bus_reduce_wide_tree(StridedRows{partials, row_stride}, n_rows, frames, scratch, counters, bus, blockIdx.x);
}

// Grouped forms for routed banks: blockIdx.x as in the kernels above, blockIdx.y = the span (bus) of the group,
// striding by gridDim.y past 65,535 spans.  One launch covers every bus of its group, however many.
__global__ void __launch_bounds__(256) bus_reduce_grouped_kernel(const BusGroup g) {
    for (uint32_t e = blockIdx.y; e < g.n_spans; e += gridDim.y) {
        const BusSpan s = g.spans[e];
        float* __restrict__ bus = g.buses + (size_t)s.bus * g.bus_stride;
        const ListedRows rows{g.rows, g.row_stride, g.idx + s.begin};
        if (s.count == 1u) {
            // a bus of one warp is that warp's partial, as a standalone one-warp bank writes it (a -0.0 stays -0.0)
            const uint32_t t = blockIdx.x * 32u + (threadIdx.x & 31u);
            if (threadIdx.x < 32u && t < g.frames) bus[t] = rows(0)[t];
        } else {
            bus_reduce_tree(rows, s.count, g.frames, bus, blockIdx.x);
        }
        __syncthreads();                                   // the shared sums are free for the next span
    }
}

__global__ void __launch_bounds__(256, 8) bus_reduce_wide_grouped_kernel(const BusGroup g, float* scratch,
                                                                      unsigned int* counters) {
    for (uint32_t e = blockIdx.y; e < g.n_spans; e += gridDim.y) {
        const BusSpan s = g.spans[e];
        bus_reduce_wide_tree(ListedRows{g.rows, g.row_stride, g.idx + s.begin}, s.count, g.frames,
                             scratch + (size_t)e * kRedSplit * g.frames, counters + (size_t)e * kBusCounters,
                             g.buses + (size_t)s.bus * g.bus_stride, blockIdx.x);
        __syncthreads();
    }
}

// Buses of up to 32 voices and several kinds (several warps): each adds its voices' rows in voice order from +0.0,
// the reference's order, as launch_ts_mix_rows does for one bank.  One thread per frame and bus.
__global__ void __launch_bounds__(256) mix_rows_grouped_kernel(const BusGroup g) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.frames) return;
    for (uint32_t e = blockIdx.y; e < g.n_spans; e += gridDim.y) {
        const BusSpan s = g.spans[e];
        const ListedRows rows{g.rows, g.row_stride, g.idx + s.begin};
        float acc = 0.0f;
        for (uint32_t r = 0; r < s.count; r++) acc = __fadd_rn(acc, rows(r)[t]);
        g.buses[(size_t)s.bus * g.bus_stride + t] = acc;
    }
}

__global__ void gather_u32_kernel(const uint32_t* __restrict__ staged, const float* __restrict__ row_index_bits,
                                  uint32_t* __restrict__ dst, uint32_t n) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const uint32_t r = __float_as_uint(row_index_bits[s]);
    if (r != kPadRow) dst[s] = staged[r];
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
template <int TRACE>
static size_t render_smem(const RenderArgs& a) {
    return (warp_smem_floats() + (TRACE == TRACE_METER ? kMeterFloats : 0)) * sizeof(float) + (a.has_sine ? 4096 : 0);
}

template <int FILTER, int TRACE>
static cudaError_t launch_t(const RenderArgs& a, cudaStream_t stream) {
    render_kernel<FILTER, TRACE><<<render_warps(a.slot_end - a.slot_begin), 32, render_smem<TRACE>(a), stream>>>(a);
    return cudaGetLastError();
}

template <int FILTER>
static cudaError_t launch_f(const RenderArgs& a, int trace, cudaStream_t stream) {
    if (trace == TRACE_PHASE) return launch_t<FILTER, TRACE_PHASE>(a, stream);
    return a.sum_sq ? launch_t<FILTER, TRACE_METER>(a, stream) : launch_t<FILTER, TRACE_NONE>(a, stream);
}

// The same launch shape and shared memory as launch_t: neither depends on the filter.
template <int TRACE>
static cudaError_t launch_mixed_t(const RenderArgs& a, cudaStream_t stream) {
    render_kernel_mixed<TRACE><<<render_warps(a.slot_end - a.slot_begin), 32, render_smem<TRACE>(a), stream>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_render(const RenderArgs& a, uint32_t filter_kind, int trace, cudaStream_t stream) {
    if (a.n_voices == 0 || a.frames == 0) return cudaSuccess;
    if (a.warp_kinds) {
        if (trace == TRACE_PHASE) return launch_mixed_t<TRACE_PHASE>(a, stream);
        return a.sum_sq ? launch_mixed_t<TRACE_METER>(a, stream) : launch_mixed_t<TRACE_NONE>(a, stream);
    }
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

static dim3 grouped_grid(uint32_t blocks, uint32_t n_spans) { return dim3(blocks, n_spans < 65535u ? n_spans : 65535u); }

cudaError_t launch_bus_reduce_grouped(const BusGroup& g, cudaStream_t stream) {
    if (g.frames == 0 || g.n_spans == 0) return cudaSuccess;
    bus_reduce_grouped_kernel<<<grouped_grid((g.frames + 31) / 32, g.n_spans), 256, 0, stream>>>(g);
    return cudaGetLastError();
}

cudaError_t launch_bus_reduce_wide_grouped(const BusGroup& g, float* scratch, unsigned int* counters, cudaStream_t stream) {
    if (g.frames == 0 || g.n_spans == 0) return cudaSuccess;
    bus_reduce_wide_grouped_kernel<<<grouped_grid(g.frames / 128u * kRedSplit, g.n_spans), 256, 0, stream>>>(g, scratch, counters);
    return cudaGetLastError();
}

cudaError_t launch_mix_rows_grouped(const BusGroup& g, cudaStream_t stream) {
    if (g.frames == 0 || g.n_spans == 0) return cudaSuccess;
    mix_rows_grouped_kernel<<<grouped_grid((g.frames + 255) / 256, g.n_spans), 256, 0, stream>>>(g);
    return cudaGetLastError();
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
