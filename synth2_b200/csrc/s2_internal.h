// s2_internal.h — shared between the kernels (s2_kernels.cu) and the C-ABI host layer (s2_capi.cu).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace s2 {

// Device-resident voice parameters: struct-of-arrays, row k at params[k * vpad + v], so the 32
// lanes of a warp (= 32 consecutive voices) load each field with one coalesced request.
// u32 fields are stored as raw bits in the float array.
enum ParamIdx {
    P_KIND = 0, P_SEED, P_PITCH, P_GAIN, P_NOISE, P_LPF, P_DAMP,
    P_AA, P_AD, P_AS, P_AR,   // amp ADSR (ms, ms, level, ms)
    P_MA, P_MD, P_MS, P_MR,   // mod ADSR
    P_AMT_OSC, P_AMT_LPF,
    P_RELEASE, P_ACTIVE,
    P_ROW,                    // caller-visible voice index of this slot (output row, see s2_capi.cu "slots")
    P_COUNT
};

// Carried state, same layout: state[k * vpad + v].
enum StateIdx {
    S_PHASE = 0, S_HAS_PHASE, S_OFFSET, S_LAST, S_X1, S_X2, S_Y1, S_Y2,
    // Memo of the constants derived from the oscillator frequency and the filter cutoff (divisions,
    // exp / sin / cos in binary64), keyed by the exact input bits: a launch that finds its key reuses
    // them instead of re-deriving ~1000 instructions per voice.  Not part of s2_voice_state.
    S_FO_KEY, S_OSC_P, S_OSC_D, S_OSC_SLOPE, S_OSC_HALF, S_OSC_TS1, S_OSC_TS2,
    S_FL_KEY, S_DAMP_KEY, S_FC_C0, S_FC_C1, S_FC_C2,
    S_COUNT
};
constexpr uint32_t kNoKey = 0x7fc00001u;   // a NaN payload no frequency can have

// TRACE_METER: a render exactly as TRACE_NONE that also accumulates the per-voice meters of RenderArgs (sum_sq, peak);
// launch_render takes it for a TRACE_NONE launch whose meters are set.
enum TraceMode { TRACE_NONE = 0, TRACE_PHASE = 1, TRACE_METER = 2 };

struct RenderArgs {
    const float* params;   // [P_COUNT][vpad]
    float* state;          // [S_COUNT][vpad]
    uint32_t n_voices;     // voices in the whole bank
    uint32_t slot_begin;   // this launch renders slots [slot_begin, slot_end): a sub-bank (multiple of 64) or the bank
    uint32_t slot_end;
    uint32_t vpad;
    float sample_rate;     // `sample_rate.0 as f32` (filters.rs:17, units.rs:21)
    uint32_t frames;       // frames to render this launch
    float* voice_out;      // [n_voices][row_stride] or nullptr
    size_t row_stride;
    float* bus_partials;   // [n_warps][frames] or nullptr
    uint32_t has_sine;     // any voice uses the table oscillator -> stage SIN_TABLE in smem
    float one;             // 1.0f, opaque to the compiler (s2_cutoff.h: vaddp)
    // A staged note-off table to apply first (pipelined banks): release offset of slot s = staged_release[caller's
    // voice index of s], also written to release_row[s] so that it persists.  nullptr = the parameter row as it is.
    const uint32_t* staged_release;
    uint32_t* release_row;
    uint32_t force_path;   // test hook (S2_FORCE_PATH): 0 = normal, 1 = moving-cutoff chunks one frame at a time,
                           // 2 = every chunk through the general per-frame path, 3 = packed moving-cutoff chunks
                           // without the lane-pair help (chunk_modcut_pk only)
    // Per-voice meters (s2_bank_render_metered), indexed by the caller's voice index, or both nullptr: every active
    // voice adds its sum of y*y over the launch's frames to sum_sq and raises peak to its largest |y| (magnitude
    // bits).  Last, so that the fields above keep their parameter offsets in the unmetered kernels.
    double* sum_sq;
    uint32_t* peak;
    // Mixed-filter banks (s2_bank_create_mixed): the filter kind of each warp of the bank (slot / 32), or nullptr for
    // a bank of one kind.  With it launch_render takes render_kernel_mixed, whatever its filter_kind argument says.
    // Last, like the meters.
    const uint8_t* warp_kinds;
};

// P_ROW of a padding slot of a mixed-filter bank: no caller voice, never active (s2_capi.cu "slots").
constexpr uint32_t kPadRow = 0xffffffffu;
// warp_kinds entry: the filter kind in the low bits, and
//   kWarpNarrowBus   the warp's bus (the whole bank, unless it is routed) has at most 32 voices, so its partial adds
//                    in voice order from +0.0 as a one-warp bank's does;
//   kWarpBusRows     routed banks rendering their buses without caller rows: the warp belongs to a bus of up to 32
//                    voices and several kinds, whose sum is added from its voices' rows, so its voices write rows to
//                    the bus scratch.  The row of each slot's voice (kPadRow: none) is a u32 array right after the
//                    table, at warp_table_bytes(vpad); the bus scratch follows the render's partial rows, at
//                    bus_partials + bus_scratch_at(vpad, frames), rows (frames + 3) & ~3 floats apart.
// (RenderArgs carries no field for these: a larger struct changes the code of the single-kind render kernels.)
constexpr uint32_t kWarpKindMask = 7u;
constexpr uint32_t kWarpNarrowBus = 8u;
constexpr uint32_t kWarpBusRows = 16u;
__host__ __device__ constexpr size_t warp_table_bytes(uint32_t vpad) { return ((size_t)(vpad / 32u) + 3u) & ~(size_t)3u; }
__host__ __device__ constexpr size_t bus_scratch_at(uint32_t vpad, uint32_t frames) {
    return ((size_t)(vpad / 32u) * frames + 3u) & ~(size_t)3u;
}

// One bus of a grouped reduction: its rows are rows + idx[begin + r] * row_stride for r < count, and it is written to
// buses + bus * bus_stride.
struct BusSpan { uint32_t bus, begin, count; };
struct BusGroup {
    const BusSpan* spans;
    uint32_t n_spans;
    const uint32_t* idx;
    const float* rows;
    size_t row_stride;
    float* buses;
    size_t bus_stride;
    uint32_t frames;
};

constexpr int kChunk = 32;          // frames per compute chunk (classification granularity)
// The render kernel's tile is 32 voices x 64 frames = two chunks: a warp then writes 256 contiguous bytes per output
// row per visit.  128 bytes per row per visit tops out at 5.1 TB/s of write bandwidth on this part whatever the
// kernel does in between, 256 bytes at 5.9 TB/s (tools/ubench/write_bw.cu, profiles/r2_write_bw.txt).
constexpr int kTileFrames = 64;
constexpr int kTileStride = 68;     // floats per tile row: 16-B aligned rows, conflict-free STS.128/LDS.128
constexpr int kTsTileStride = 36;   // the time-split kernel's 32-frame tile

// Launchers (s2_kernels.cu).  Return the cudaError_t of the launch.  A warp renders 32 consecutive slots.
cudaError_t launch_render(const RenderArgs& a, uint32_t filter_kind, int trace, cudaStream_t stream);
uint32_t render_warps(uint32_t n_voices);
// time-split rendering of narrow banks (s2_kernel_ts.cu): the phase pre-pass writes, for each of the block's 32
// time segments, the phase of its first frame and of the two frames before it to seg_phase[n_voices][3][32];
// the render consumes it.
// frames must be a multiple of 1024.
cudaError_t launch_ts_phase(const RenderArgs& a, float* seg_phase, cudaStream_t stream);
// moving: some voice's cutoff follows a ramping mod envelope in this block (per-frame coefficients)
cudaError_t launch_ts_render(const RenderArgs& a, uint32_t filter_kind, bool moving, const float* seg_phase,
                             cudaStream_t stream);
// bus[t] = sum of rows[r * row_stride + t] over r = 0, 1, ..., n_rows - 1, sequentially from +0.0 (the reference's
// order; for banks of at most 32 voices)
cudaError_t launch_ts_mix_rows(const float* rows, uint32_t n_rows, size_t row_stride, uint32_t frames, float* bus,
                               cudaStream_t stream);
// one kernel, fixed summation order; partial row w starts at partials + w * row_stride.  With `counters` (kBusCounters
// zeroed words owned by the bank, launches on one stream at a time) and `scratch` of bus_scratch_floats(n_warps,
// frames) floats, wide banks take the four-frames-per-lane form.
constexpr uint32_t kBusCounters = 1024;
cudaError_t launch_bus_reduce(const float* partials, uint32_t n_warps, size_t row_stride, uint32_t frames, float* bus,
                              cudaStream_t stream, unsigned int* counters = nullptr, float* scratch = nullptr);
// floats of scratch the four-frames-per-lane form reads for this shape; 0 where that form does not apply
size_t bus_scratch_floats(uint32_t n_rows, uint32_t frames);
// Grouped reductions of routed banks: one launch for every bus of the group, each bus summed exactly as the launcher
// above sums a standalone bank's rows.  launch_bus_reduce_grouped: the one-frame-per-lane form (a bus of one row is
// a copy of it, a bus of none is +0.0).  launch_bus_reduce_wide_grouped: the four-frames-per-lane form, for buses
// that pass its tests; span e uses scratch + e * bus_scratch_floats and counters + e * kBusCounters.
// launch_mix_rows_grouped: each bus adds its rows sequentially from +0.0, as launch_ts_mix_rows does.
cudaError_t launch_bus_reduce_grouped(const BusGroup& g, cudaStream_t stream);
cudaError_t launch_bus_reduce_wide_grouped(const BusGroup& g, float* scratch, unsigned int* counters, cudaStream_t stream);
cudaError_t launch_mix_rows_grouped(const BusGroup& g, cudaStream_t stream);
// release_row[slot] = staged[voice_of_slot[slot]]  (bulk note-off table given in voice order)
cudaError_t launch_gather_u32(const uint32_t* staged, const float* row_index_bits, uint32_t* dst_row,
                              uint32_t n, cudaStream_t stream);
// Bulk note-on (s2_bank_set_voices).  `batch` holds m entries column-major: [P_COUNT][m] parameters, [S_COUNT][m] fresh
// state, then [m] target slots (u32 bits).  Entries [begin, begin + count) are written to their slots of params /
// state; with `staged_release` (a pending note-off table in voice order) also staged_release[P_ROW] = P_RELEASE.
cudaError_t launch_set_voices(const float* batch, uint32_t m, uint32_t begin, uint32_t count, float* params,
                              float* state, uint32_t vpad, uint32_t* staged_release, cudaStream_t stream);

}  // namespace s2
