// s2_capi.cu — host side of libs2cuda.so: the C ABI declared in include/s2_cuda.h.
//
// Two objects:
//   s2_bank  — V voices resident on one GPU (SoA parameters + carried state), rendered by
//              s2::launch_render; the batched form of process::process_layer_buf_simd.
//   s2_synth — mirror of synth::Synth (s2_lib/src/try3/synth.rs): 8 voice slots, the default
//              patch, oldest-voice allocation, note_on / note_off / sample.  The voice bookkeeping
//              runs on the host exactly like the reference's; only rendering goes to the GPU.
// No CPU rendering exists in this library.
#include "../../include/s2_cuda.h"
#include "s2_internal.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
}  // namespace

namespace s2 {
// fills s2_last_error(); also the error reporting of the other host translation units of the library (s2_patch.cpp)
int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
}  // namespace s2

namespace {

constexpr auto fail = s2::set_error;

#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail(S2_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                \
    } while (0)

bool finite_nonneg(float x) { return std::isfinite(x) && x >= 0.0f; }

int validate_voice(const s2_voice_desc& d, size_t index, uint32_t filter_kind = S2_FILTER_ONE_POLE) {
    // second-order filters: damping (band-pass: the quality factor) divides or scales the coefficients
    // (dsp_filters.rs:99-109, 197-207; 0.2 is the documented minimum, :94-96); zero gives tan(inf) / a zero denominator
    if (filter_kind >= S2_FILTER_BIQUAD_LP && filter_kind <= S2_FILTER_BIQUAD_BP && !(d.damping > 0.0f))
        return fail(S2_ERR_INVALID, "voice %zu: damping must be > 0 for the second-order filters", index);
    if (d.osc_kind > S2_OSC_SINE) return fail(S2_ERR_INVALID, "voice %zu: osc_kind %u", index, d.osc_kind);
    if (!(std::isfinite(d.pitch_hz) && d.pitch_hz > 0.0f))
        return fail(S2_ERR_INVALID, "voice %zu: pitch_hz must be finite and > 0", index);
    if (!(std::isfinite(d.lpf_freq_hz) && d.lpf_freq_hz >= 0.0f))
        return fail(S2_ERR_INVALID, "voice %zu: lpf_freq_hz must be finite and >= 0", index);
    const float ms[6] = {d.amp_attack_ms, d.amp_decay_ms, d.amp_release_ms,
                         d.mod_attack_ms, d.mod_decay_ms, d.mod_release_ms};
    for (float m : ms)
        if (!finite_nonneg(m)) return fail(S2_ERR_INVALID, "voice %zu: envelope times must be finite and >= 0", index);
    const float fl[7] = {d.osc_gain, d.noise_amt, d.damping, d.amp_sustain, d.mod_sustain,
                         d.mod_env_to_osc_freq, d.mod_env_to_lpf_freq};
    for (float f : fl)
        if (!std::isfinite(f)) return fail(S2_ERR_INVALID, "voice %zu: non-finite parameter", index);
    return S2_OK;
}

uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
float ubits(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }

void pack_voice(const s2_voice_desc& d, uint32_t row, float* col, size_t pitch) {
    using namespace s2;
    col[P_ROW * pitch] = ubits(row);
    col[P_KIND * pitch] = ubits(d.osc_kind);
    col[P_SEED * pitch] = ubits(d.noise_seed);
    col[P_PITCH * pitch] = d.pitch_hz;
    col[P_GAIN * pitch] = d.osc_gain;
    col[P_NOISE * pitch] = d.noise_amt;
    col[P_LPF * pitch] = d.lpf_freq_hz;
    col[P_DAMP * pitch] = d.damping;
    col[P_AA * pitch] = d.amp_attack_ms;
    col[P_AD * pitch] = d.amp_decay_ms;
    col[P_AS * pitch] = d.amp_sustain;
    col[P_AR * pitch] = d.amp_release_ms;
    col[P_MA * pitch] = d.mod_attack_ms;
    col[P_MD * pitch] = d.mod_decay_ms;
    col[P_MS * pitch] = d.mod_sustain;
    col[P_MR * pitch] = d.mod_release_ms;
    col[P_AMT_OSC * pitch] = d.mod_env_to_osc_freq;
    col[P_AMT_LPF * pitch] = d.mod_env_to_lpf_freq;
    col[P_RELEASE * pitch] = ubits(d.release_offset);
    col[P_ACTIVE * pitch] = ubits(d.active ? 1u : 0u);
}

void pack_state(const s2_voice_state& s, float* col, size_t pitch) {
    using namespace s2;
    col[S_PHASE * pitch] = s.phase;
    col[S_HAS_PHASE * pitch] = ubits(s.has_phase ? 1u : 0u);
    col[S_OFFSET * pitch] = ubits(s.frame_offset);
    col[S_LAST * pitch] = s.lpf_last;
    col[S_X1 * pitch] = s.x1;
    col[S_X2 * pitch] = s.x2;
    col[S_Y1 * pitch] = s.y1;
    col[S_Y2 * pitch] = s.y2;
    // derived-constant memo: empty (the kernel re-derives and refills it)
    for (int k = S_FO_KEY; k < S_COUNT; k++) col[k * pitch] = 0.0f;
    col[S_FO_KEY * pitch] = ubits(kNoKey);
    col[S_FL_KEY * pitch] = ubits(kNoKey);
}

// A note-on: the voice's parameter column and a fresh state (st::Layer::default(), synth.rs:68) at its frame offset.
void pack_note_on(const s2_voice_desc& d, uint32_t index, float* pcol, float* scol, size_t pitch) {
    pack_voice(d, index, pcol, pitch);
    s2_voice_state st;
    memset(&st, 0, sizeof st);
    st.frame_offset = d.frame_offset;
    pack_state(st, scol, pitch);
}

struct VoiceBook {           // host mirror of what the device will hold, O(1) per render
    uint32_t start_offset;   // frame offset when the voice was (re)started
    uint64_t start_total;    // bank->total_frames at that moment
    uint32_t active;
    uint32_t osc_kind;
};

// Partial-sum buffers of the pipelined mix.  The reduction of step i runs on the (high-priority) mix stream
// while the sub-banks already render step i+1; with only two buffers step i+2 would have to wait for it,
// and a reduction that is slow to get SM slots next to the render blocks then stalls the whole pipeline.
constexpr int kMixBufs = 4;
constexpr int kTsBufs = 4;                 // the phase pre-pass may run this many blocks ahead of the renders
constexpr size_t kTsMaxVoices = 16384;     // beyond this a bank fills the machine with one voice per lane

cudaError_t make_event(cudaEvent_t& e) { return e ? cudaSuccess : cudaEventCreateWithFlags(&e, cudaEventDisableTiming); }
void destroy(cudaEvent_t e) { if (e) cudaEventDestroy(e); }
void destroy(cudaStream_t s) { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } }

// Pipelined mode (s2_bank_set_pipeline): the bank is cut into n_sub contiguous slot ranges, each rendered on its
// own internal stream.  Consecutive render calls then overlap across sub-banks (no device-wide barrier between
// blocks), which keeps every SM sub-partition supplied with warps while the slower ones finish
// (profiles/r1_notes.md: +14 % at 65,536 voices).
struct Pipeline {
    cudaStream_t sub[8] = {};
    cudaStream_t mix = nullptr;           // bus reduction and copies of the pipelined mode
    cudaStream_t upload = nullptr;        // note-off table uploads (independent of the mix stream)
    cudaEvent_t ev_gather[8][2] = {};     // sub-bank k has applied the table staged in buffer q
    cudaEvent_t ev_sub[8] = {};           // last work issued on sub-stream k
    cudaEvent_t ev_mix[kMixBufs] = {};    // reduction of partial buffer p finished
    cudaEvent_t ev_stage[2] = {};         // note-off table p has landed in its staging buffer
    cudaEvent_t ev_tail = nullptr;        // last work issued on the mix stream
    // Staging of the bulk note-off table, in voice order.  Buffer 0 also serves s2_bank_set_releases of a bank on
    // one stream whose slots are permuted.
    uint32_t* d_staging[2] = {};
    float* d_partials[kMixBufs] = {};
    size_t partials_cap = 0;              // floats, each of the kMixBufs buffers
    uint64_t step = 0, table_step = 0;
    int table_pending = -1;               // staging buffer index holding a table not yet applied, or -1

    // What n_sub ranges need, created once and kept when the bank goes back to fewer ranges.
    int create(int n_sub, size_t n_voices) {
        for (int k = 0; k < n_sub; k++) {
            if (!sub[k]) CUDA_TRY(cudaStreamCreateWithFlags(&sub[k], cudaStreamNonBlocking));
            CUDA_TRY(make_event(ev_sub[k]));
            CUDA_TRY(cudaEventRecord(ev_sub[k], sub[k]));
        }
        if (!mix) {
            int prio_lo = 0, prio_hi = 0;
            CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            CUDA_TRY(cudaStreamCreateWithPriority(&mix, cudaStreamNonBlocking, prio_hi));
        }
        if (!upload) CUDA_TRY(cudaStreamCreateWithFlags(&upload, cudaStreamNonBlocking));
        for (int k = 0; k < n_sub; k++)
            for (int q = 0; q < 2; q++)
                if (!ev_gather[k][q]) {
                    CUDA_TRY(make_event(ev_gather[k][q]));
                    CUDA_TRY(cudaEventRecord(ev_gather[k][q], sub[k]));
                }
        for (int i = 0; i < kMixBufs; i++) CUDA_TRY(make_event(ev_mix[i]));
        for (int i = 0; i < 2; i++) {
            CUDA_TRY(make_event(ev_stage[i]));
            if (!d_staging[i]) CUDA_TRY(cudaMalloc(&d_staging[i], n_voices * sizeof(uint32_t)));
        }
        CUDA_TRY(make_event(ev_tail));
        return S2_OK;
    }

    void release() {
        for (int k = 0; k < 8; k++) {
            destroy(sub[k]);
            destroy(ev_sub[k]);
            for (int q = 0; q < 2; q++) destroy(ev_gather[k][q]);
        }
        destroy(mix);
        destroy(upload);
        destroy(ev_tail);
        for (int i = 0; i < 2; i++) { destroy(ev_stage[i]); cudaFree(d_staging[i]); }
        for (int i = 0; i < kMixBufs; i++) { destroy(ev_mix[i]); cudaFree(d_partials[i]); }
    }
};

// Staging of s2_bank_set_voices: batch i is packed into page-locked buffer r = i % kBatchBufs, sent with one copy to
// device buffer r and scattered from there, so the caller's arrays are free on return and the copy never waits for
// a pageable-memory bounce.  Buffer r is reused once its copy (host side) and its scatters (device side) have run.
constexpr int kBatchBufs = 4;

struct VoiceBatches {
    float* h[kBatchBufs] = {};             // page-locked
    float* d[kBatchBufs] = {};
    size_t h_cap = 0, d_cap = 0;           // floats, each buffer
    cudaEvent_t ev_copied[kBatchBufs] = {};    // the copy out of h[r] has finished
    cudaEvent_t ev_read[kBatchBufs][8] = {};   // voice range k's scatter out of d[r] has finished (pipelined)
    uint64_t next = 0;
    std::vector<uint32_t> stamp;           // per voice: the batch generation that last kept an entry of it
    uint32_t gen = 0;

    int create() {
        for (int r = 0; r < kBatchBufs; r++) {
            CUDA_TRY(make_event(ev_copied[r]));
            for (int k = 0; k < 8; k++) CUDA_TRY(make_event(ev_read[r][k]));
        }
        return S2_OK;
    }

    void release() {
        for (int r = 0; r < kBatchBufs; r++) {
            destroy(ev_copied[r]);
            for (int k = 0; k < 8; k++) destroy(ev_read[r][k]);
            if (h[r]) cudaFreeHost(h[r]);
            cudaFree(d[r]);
        }
    }
};

// Time-split mode (s2_bank_set_time_split, s2_kernel_ts.cu): narrow one-pole banks render a block as 32 time
// segments per voice.  The phase pre-pass runs on its own stream, ahead of the renders.
struct TimeSplit {
    bool enabled = false;
    bool main_dirty = true;               // b->stream carries state writes the pre-pass stream has not seen
    cudaStream_t stream = nullptr;        // the phase pre-pass
    float* d_seg_phase[kTsBufs] = {};     // [n_slots][3][32] segment-start phases (and the two before) of block p
    cudaEvent_t ev_k1[kTsBufs] = {}, ev_k2[kTsBufs] = {}, ev_main = nullptr;
    uint64_t step = 0, blocks = 0;        // blocks: blocks rendered through the time-split kernels
    std::vector<s2_voice_desc> descs;     // host copy of the voice descriptions (banks <= kTsMaxVoices only)

    int create(size_t n_slots) {
        if (!stream) CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        for (int i = 0; i < kTsBufs; i++) {
            if (!d_seg_phase[i]) CUDA_TRY(cudaMalloc(&d_seg_phase[i], n_slots * 96 * sizeof(float)));
            CUDA_TRY(make_event(ev_k1[i]));
            CUDA_TRY(make_event(ev_k2[i]));
        }
        CUDA_TRY(make_event(ev_main));
        return S2_OK;
    }

    void release() {
        destroy(stream);
        for (int i = 0; i < kTsBufs; i++) { destroy(ev_k1[i]); destroy(ev_k2[i]); cudaFree(d_seg_phase[i]); }
        destroy(ev_main);
    }
};

// Routed banks (s2_bank_create_routed): what the grouped bus reductions read, in one device array of 32-bit words.
// Each bus's rows are listed once: its voices in voice order (rows of the caller, or of the time-split path) and its
// warps in the order of a standalone bank of its voices (partial rows).  A group of spans (s2::BusSpan) is the buses
// of one reduction form, each pointing into one of those lists.
struct Routes {
    uint32_t* d = nullptr;
    // word offsets into d
    size_t voices = 0, warps = 0, iota = 0;
    size_t rows_voice = 0, rows_scratch = 0, partial = 0, ts_narrow = 0, ts_wide = 0;
    // spans per group.  partial: n_rest buses, then the n_big of >= 512 warps that the four-frames-per-lane form
    // may take
    uint32_t n_rows = 0, n_rest = 0, n_big = 0, n_ts_narrow = 0, n_ts_wide = 0;
    uint32_t n_scratch = 0;    // voices of the buses added from their rows (one bus-scratch row each)

    const s2::BusSpan* spans(size_t off) const { return reinterpret_cast<const s2::BusSpan*>(d + off); }
};

}  // namespace

struct s2_bank {
    int device = 0;
    cudaStream_t stream = nullptr;
    uint32_t sample_rate = 0;
    uint32_t filter_kind = 0;    // the kind of every voice, or of voice 0 of a mixed-filter bank
    size_t n_voices = 0;
    size_t n_slots = 0;          // n_voices plus the padding slots of a mixed-filter bank
    size_t vpad = 0;
    float* d_params = nullptr;
    float* d_state = nullptr;
    float* d_partials = nullptr;
    size_t partials_cap = 0;     // floats
    unsigned int* d_bus_counters = nullptr;   // s2::kBusCounters zeroed words of the wide bus reduction per bus that
                                              // may take it (one for a bank that is not routed)
    float* d_bus = nullptr;
    size_t bus_cap = 0;          // floats
    std::vector<VoiceBook> book;  // indexed by voice
    // "Slots": device arrays are indexed by slot, not by the caller's voice index.  Banks wider than
    // one warp are sorted by (active, oscillator kind, when the amp envelope rests) at creation so that the
    // 32 lanes of a warp run the same code for as long as possible, then dealt over the voice ranges; output
    // rows, state get/set and per-voice calls keep the caller's indices.  Banks of <= 32 voices keep
    // the identity order, which also keeps the bus sum in the reference's voice order.
    // Mixed-filter banks: kinds are grouped, each group but the last padded to whole warps of 32 slots with padding
    // slots (voice_of_slot = P_ROW = kPadRow, inactive).
    std::vector<uint32_t> slot_of_voice, voice_of_slot;
    bool identity = true;
    std::vector<uint32_t> voice_kind;   // filter kind of each voice
    uint32_t n_kinds = 1;               // distinct kinds; above 1 the render takes the mixed kernel
    uint8_t* d_warp_kinds = nullptr;    // [n_slots / 32 rounded up] filter kind and flags of each warp (s2::kWarpNarrowBus)
    // Routed banks: n_buses > 1, the bus of every voice, and the lists of their bus reductions.  A bank made any
    // other way has one bus, and bus_of_voice is empty.
    uint32_t n_buses = 1;
    std::vector<uint32_t> bus_of_voice;
    Routes route;
    uint32_t force_path = 0;      // test hook (S2_FORCE_PATH, see RenderArgs)
    int n_sub = 1;                // voice ranges of the pipelined mode; 1 = everything on the bank's stream
    Pipeline pipe;
    TimeSplit split;
    VoiceBatches batches;
    uint64_t total_frames = 0;
    uint64_t max_offset = 0;     // upper bound of any active voice's frame offset
    size_t n_sine = 0;
};

namespace {

uint32_t current_offset(const s2_bank* b, size_t i) {
    const VoiceBook& vb = b->book[i];
    if (!vb.active) return vb.start_offset;
    const uint64_t o = (uint64_t)vb.start_offset + (b->total_frames - vb.start_total);
    return o > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)o;   // saturating_add, synth.rs:197
}

// The host mirrors of a voice replaced by s2_bank_set_voice(s), updated at call time in call order.
void note_voice(s2_bank* b, size_t index, const s2_voice_desc& d) {
    if (b->book[index].osc_kind == S2_OSC_SINE) b->n_sine--;
    if (d.osc_kind == S2_OSC_SINE) b->n_sine++;
    b->book[index] = {d.frame_offset, b->total_frames, d.active ? 1u : 0u, d.osc_kind};
    if (!b->split.descs.empty()) b->split.descs[index] = d;
    if (d.active && d.frame_offset > b->max_offset) b->max_offset = d.frame_offset;
}

// Waits (on the host) for everything the bank has issued on its internal streams.
int bank_drain(s2_bank* b) {
    for (int k = 0; k < b->n_sub && b->n_sub > 1; k++) CUDA_TRY(cudaStreamSynchronize(b->pipe.sub[k]));
    if (b->pipe.mix) CUDA_TRY(cudaStreamSynchronize(b->pipe.mix));
    if (b->pipe.upload) CUDA_TRY(cudaStreamSynchronize(b->pipe.upload));
    if (b->split.stream) CUDA_TRY(cudaStreamSynchronize(b->split.stream));
    return S2_OK;
}

// Grows the n device buffers bufs[0..n) (pinned: page-locked host buffers) to `need` floats each; they share the
// capacity `cap`.  The bank's internal streams may still use the old buffers, so the bank (if any) is drained before
// they are freed.  A failed allocation leaves that buffer null and cap 0.
int grow(s2_bank* b, float** bufs, int n, size_t& cap, size_t need, bool pinned = false) {
    if (need <= cap) return S2_OK;
    if (b) { int rc = bank_drain(b); if (rc) return rc; }
    for (int i = 0; i < n; i++) {
        if (bufs[i]) CUDA_TRY(pinned ? cudaFreeHost(bufs[i]) : cudaFree(bufs[i]));
        bufs[i] = nullptr;
    }
    cap = 0;
    for (int i = 0; i < n; i++)
        CUDA_TRY(pinned ? cudaMallocHost(&bufs[i], need * sizeof(float)) : cudaMalloc(&bufs[i], need * sizeof(float)));
    cap = need;
    return S2_OK;
}

// A note-off table staged for the next pipelined render (s2_bank_set_releases) is applied by that render's kernels.
// An entry that writes the release row itself, renders outside the voice ranges or changes the ranges applies it
// here first, on the bank's stream, so that edits take effect in call order.  Call after bank_drain.
int apply_staged_table(s2_bank* b) {
    Pipeline& pl = b->pipe;
    if (b->n_sub <= 1 || pl.table_pending < 0) return S2_OK;
    CUDA_TRY(cudaStreamWaitEvent(b->stream, pl.ev_stage[pl.table_pending], 0));
    CUDA_TRY(s2::launch_gather_u32(pl.d_staging[pl.table_pending], b->d_params + (size_t)s2::P_ROW * b->vpad,
                                   reinterpret_cast<uint32_t*>(b->d_params + (size_t)s2::P_RELEASE * b->vpad),
                                   (uint32_t)b->n_slots, b->stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaStreamSynchronize(b->stream));   // the staging buffer is free again before the next upload
    pl.table_pending = -1;
    return S2_OK;
}

// Before an entry that works on the bank's stream alone: every edit made so far is then on that stream, in call order.
int settle_edits(s2_bank* b) {
    int rc = bank_drain(b);
    return rc ? rc : apply_staged_table(b);
}

// Every RenderArgs field from the bank, for the whole slot range, without bus partials or a staged table.  A plain
// render is a metered one with null meters.
s2::RenderArgs base_args(const s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, double* d_sum_sq,
                         uint32_t* d_peak) {
    s2::RenderArgs a;
    a.params = b->d_params;
    a.state = b->d_state;
    a.n_voices = (uint32_t)b->n_voices;
    a.slot_begin = 0;
    a.slot_end = (uint32_t)b->n_slots;
    a.vpad = (uint32_t)b->vpad;
    a.sample_rate = (float)b->sample_rate;
    a.frames = (uint32_t)frames;
    a.voice_out = d_voice_out;
    a.row_stride = row_stride;
    a.bus_partials = nullptr;
    a.has_sine = b->n_sine ? 1u : 0u;
    a.one = 1.0f;
    a.force_path = b->force_path;
    a.staged_release = nullptr;
    a.release_row = nullptr;
    a.sum_sq = d_sum_sq;
    a.peak = d_peak;
    a.warp_kinds = b->d_warp_kinds;
    return a;
}

// Floats of a partial-sum buffer: one row of `frames` per warp, then the scratch of the wide bus reduction.
size_t partials_floats(uint32_t n_warps, size_t frames) {
    return (size_t)n_warps * frames + s2::bus_scratch_floats(n_warps, (uint32_t)frames);
}

// The bus from the partial rows the render's warps wrote (partials_floats layout), on `st`.  A single warp's row is
// the bus: the default path renders it straight there (partials == bus), the pipelined path copies it.
int mix_partials(const s2_bank* b, float* partials, uint32_t n_warps, size_t frames, float* bus, cudaStream_t st) {
    if (partials == bus) return S2_OK;
    if (n_warps == 1) {
        CUDA_TRY(cudaMemcpyAsync(bus, partials, frames * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return S2_OK;
    }
    CUDA_TRY(s2::launch_bus_reduce(partials, n_warps, frames, (uint32_t)frames, bus, st, b->d_bus_counters,
                                   partials + (size_t)n_warps * frames));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return S2_OK;
}

// Banks of up to 32 voices that span several warps (one per kind, or per bus of a routed bank).  Their bus is added
// from the rows, in voice order from +0.0 as a one-warp bank adds it, after the render: into `a` go the caller's rows,
// or else a scratch of n_voices rows of `frames` rounded up to 16 bytes in `scratch`.
bool bus_from_rows(const s2_bank* b) { return b->n_voices <= 32 && b->n_slots > 32; }
size_t scratch_row_stride(size_t frames) { return (frames + 3) & ~(size_t)3; }

void rows_for_bus(s2::RenderArgs& a, float* scratch, size_t frames) {
    if (a.voice_out) return;
    a.voice_out = scratch;
    a.row_stride = scratch_row_stride(frames);
}

int mix_rows(const s2_bank* b, const s2::RenderArgs& a, size_t frames, float* bus, cudaStream_t st) {
    CUDA_TRY(s2::launch_ts_mix_rows(a.voice_out, (uint32_t)b->n_voices, a.row_stride, (uint32_t)frames, bus, st));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return S2_OK;
}

// The buses of a routed bank (s2_bank_render_buses).  A render's partial-sum buffer holds the warps' partial rows,
// then (at s2::bus_scratch_at) the bus scratch rows of the buses added from their voices' rows, then the scratch of
// the four-frames-per-lane form for each bus that takes it.
size_t route_wide_floats(size_t frames) { return s2::bus_scratch_floats(512u, (uint32_t)frames); }   // per bus, 0 = none
size_t route_wide_at(const s2_bank* b, size_t frames) {
    return s2::bus_scratch_at((uint32_t)b->vpad, (uint32_t)frames) + (size_t)b->route.n_scratch * scratch_row_stride(frames);
}
size_t route_floats(const s2_bank* b, size_t frames) {
    return route_wide_at(b, frames) + b->route.n_big * route_wide_floats(frames);
}

// The render writes partial rows into `partials`, and without caller rows the bus scratch rows too: the warp table
// with kWarpBusRows set, which the bank keeps after the plain one.
void route_args(const s2_bank* b, s2::RenderArgs& a, float* partials) {
    a.bus_partials = partials;
    if (!a.voice_out && b->route.n_scratch) a.warp_kinds = b->d_warp_kinds + s2::warp_table_bytes((uint32_t)b->vpad);
}

// Every bus from one render's partial rows, with the rule of a standalone bank of the bus's voices (mix_partials,
// mix_rows): one launch per reduction form present, whatever the number of buses.
int route_mix(const s2_bank* b, const s2::RenderArgs& a, size_t frames, float* d_buses, size_t bus_stride, cudaStream_t st) {
    const Routes& R = b->route;
    const bool wide = route_wide_floats(frames) != 0;
    s2::BusGroup g{};
    g.frames = (uint32_t)frames;
    g.buses = d_buses;
    g.bus_stride = bus_stride;
    g.rows = a.bus_partials;
    g.row_stride = frames;
    g.idx = R.d + R.warps;
    g.spans = R.spans(R.partial);
    g.n_spans = R.n_rest + (wide ? 0u : R.n_big);
    int n = 0;
    if (g.n_spans) { CUDA_TRY(s2::launch_bus_reduce_grouped(g, st)); n++; }
    if (wide && R.n_big) {
        g.spans = R.spans(R.partial) + R.n_rest;
        g.n_spans = R.n_big;
        CUDA_TRY(s2::launch_bus_reduce_wide_grouped(g, a.bus_partials + route_wide_at(b, frames), b->d_bus_counters, st));
        n++;
    }
    if (R.n_rows) {
        const bool scratch = a.voice_out == nullptr;
        g.rows = scratch ? a.bus_partials + s2::bus_scratch_at((uint32_t)b->vpad, (uint32_t)frames) : a.voice_out;
        g.row_stride = scratch ? scratch_row_stride(frames) : a.row_stride;
        g.idx = R.d + (scratch ? R.iota : R.voices);
        g.spans = R.spans(scratch ? R.rows_scratch : R.rows_voice);
        g.n_spans = R.n_rows;
        CUDA_TRY(s2::launch_mix_rows_grouped(g, st));
        n++;
    }
    g_launches.fetch_add(n, std::memory_order_relaxed);
    return S2_OK;
}

uint32_t sub_begin(const s2_bank* b, int k) {
    // contiguous slot ranges, multiples of 64 slots so that warps (32 or 64 slots) never straddle two
    const uint64_t groups = (b->n_slots + 63) / 64;
    const uint64_t g = groups * (uint64_t)k / (uint64_t)b->n_sub;
    const uint64_t s = g * 64;
    return (uint32_t)(s < b->n_slots ? s : b->n_slots);
}

int bank_render_pipelined(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_bus_out,
                          double* d_sum_sq, uint32_t* d_peak, float* d_buses, size_t bus_stride) {
    Pipeline& pl = b->pipe;
    const uint32_t n_warps = s2::render_warps((uint32_t)b->n_slots);
    const int p = (int)(pl.step % (uint64_t)kMixBufs);
    s2::RenderArgs a = base_args(b, frames, d_voice_out, row_stride, d_sum_sq, d_peak);
    if (d_buses) {
        int rc = grow(b, pl.d_partials, kMixBufs, pl.partials_cap, route_floats(b, frames));
        if (rc) return rc;
        route_args(b, a, pl.d_partials[p]);
    } else if (d_bus_out) {
        const size_t need = bus_from_rows(b) ? b->n_voices * scratch_row_stride(frames) : partials_floats(n_warps, frames);
        int rc = grow(b, pl.d_partials, kMixBufs, pl.partials_cap, need);
        if (rc) return rc;
        if (bus_from_rows(b)) rows_for_bus(a, pl.d_partials[p], frames);
        else a.bus_partials = pl.d_partials[p];
    }
    uint32_t* release_row = reinterpret_cast<uint32_t*>(b->d_params + (size_t)s2::P_RELEASE * b->vpad);
    for (int k = 0; k < b->n_sub; k++) {
        a.slot_begin = sub_begin(b, k);
        a.slot_end = sub_begin(b, k + 1);
        if (a.slot_begin >= a.slot_end) continue;
        cudaStream_t sk = pl.sub[k];
        if (pl.table_pending >= 0) {
            // the staged note-off table: this sub-bank's render applies it to its own slots first (kernel prologue),
            // ordered between its own renders
            CUDA_TRY(cudaStreamWaitEvent(sk, pl.ev_stage[pl.table_pending], 0));
            a.staged_release = pl.d_staging[pl.table_pending];
            a.release_row = release_row;
        }
        if ((d_bus_out || d_buses) && pl.step >= (uint64_t)kMixBufs) CUDA_TRY(cudaStreamWaitEvent(sk, pl.ev_mix[p], 0));   // partials[p] are free again
        CUDA_TRY(s2::launch_render(a, b->filter_kind, s2::TRACE_NONE, sk));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if (pl.table_pending >= 0) CUDA_TRY(cudaEventRecord(pl.ev_gather[k][pl.table_pending], sk));   // staging buffer read
        CUDA_TRY(cudaEventRecord(pl.ev_sub[k], sk));
    }
    pl.table_pending = -1;
    if (d_bus_out || d_buses) {
        for (int k = 0; k < b->n_sub; k++) CUDA_TRY(cudaStreamWaitEvent(pl.mix, pl.ev_sub[k], 0));
        int rc = d_buses ? route_mix(b, a, frames, d_buses, bus_stride, pl.mix)
                 : bus_from_rows(b) ? mix_rows(b, a, frames, d_bus_out, pl.mix)
                                    : mix_partials(b, a.bus_partials, n_warps, frames, d_bus_out, pl.mix);
        if (rc) return rc;
        CUDA_TRY(cudaEventRecord(pl.ev_mix[p], pl.mix));
    }
    pl.step++;
    b->total_frames += frames;
    b->max_offset += frames;
    return S2_OK;
}

// units.rs:44-53 in host f32 arithmetic (IEEE, no contraction: same bits as the device's make_env)
float host_ms_as_samples(float ms, float sr) { return sr * (ms / 1000.0f); }

// May this block go through the time-split kernels?  Every active voice must keep one period for the whole
// block (no pitch modulation).  Returns 0 = no, 1 = yes and every cutoff rests too (mod envelope unused by the
// cutoff, or in sustain / end until the block ends), 2 = yes but some cutoff follows a ramping mod envelope
// (per-frame coefficients).  Conservative: anything unsure renders the general way.
int ts_block_class(const s2_bank* b, size_t frames, const float* d_voice_out, bool metered) {
    if (!b->split.enabled || !d_voice_out) return 0;                            // the mix is summed from the rows
    if (metered) return 0;                                                      // the time-split kernels have no meters
    if (frames < 1024 || (frames & 1023u) != 0 || frames > (1u << 24)) return 0;   // 32 segments of whole chunks
    const float sr = (float)b->sample_rate;
    int cls = 1;
    for (size_t i = 0; i < b->n_voices; i++) {
        if (!b->book[i].active) continue;
        const s2_voice_desc& d = b->split.descs[i];
        if (d.mod_env_to_osc_freq != 0.0f) return 0;
        const uint64_t n0 = current_offset(b, i);
        if (n0 + frames > (1ull << 24)) return 0;
        const float P = sr / d.pitch_hz;
        const float step = 1.0f / P;
        if (!(step < 1.0f && P > 1.0f)) return 0;
        if (d.mod_env_to_lpf_freq != 0.0f) {
            const float A = host_ms_as_samples(d.mod_attack_ms, sr), D = host_ms_as_samples(d.mod_decay_ms, sr);
            const float R = host_ms_as_samples(d.mod_release_ms, sr);
            const float AD = A + D;
            const float Rs = fmaxf((float)d.release_offset, AD);
            const float E = Rs + R;
            const float x0 = (float)(uint32_t)n0, x1 = (float)(uint32_t)(n0 + frames - 1);
            const bool rest_sustain = x0 >= A && x0 >= AD && x1 < Rs;     // stage 2 from first to last frame
            const bool rest_end = x0 >= A && x0 >= AD && x0 >= Rs && x0 >= E;
            if (!(rest_sustain || rest_end)) cls = 2;
        }
    }
    return cls;
}

int bank_render_time_split(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_bus_out,
                           bool moving, float* d_buses, size_t bus_stride) {
    TimeSplit& ts = b->split;
    const int p = (int)(ts.step % (uint64_t)kTsBufs);
    const s2::RenderArgs a = base_args(b, frames, d_voice_out, row_stride, nullptr, nullptr);
    if (ts.main_dirty) {
        // the pre-pass reads the carried phase: order it after whatever the bank's stream wrote
        CUDA_TRY(cudaEventRecord(ts.ev_main, b->stream));
        CUDA_TRY(cudaStreamWaitEvent(ts.stream, ts.ev_main, 0));
        ts.main_dirty = false;
    }
    if (ts.step >= (uint64_t)kTsBufs) CUDA_TRY(cudaStreamWaitEvent(ts.stream, ts.ev_k2[p], 0));   // seg_phase[p] is free again
    CUDA_TRY(s2::launch_ts_phase(a, ts.d_seg_phase[p], ts.stream));
    CUDA_TRY(cudaEventRecord(ts.ev_k1[p], ts.stream));
    CUDA_TRY(cudaStreamWaitEvent(b->stream, ts.ev_k1[p], 0));
    CUDA_TRY(s2::launch_ts_render(a, b->filter_kind, moving, ts.d_seg_phase[p], b->stream));
    CUDA_TRY(cudaEventRecord(ts.ev_k2[p], b->stream));
    g_launches.fetch_add(2, std::memory_order_relaxed);
    if (d_bus_out) {
        // one warp rendered one voice: the output rows (silent voices included, as zeros) are the partial sums.
        // Up to 32 voices they are added in voice order, as on the default path; wider banks take the reduction
        // kernel's fixed tree (its one-frame-per-lane form, which needs no scratch).
        const uint32_t nv = (uint32_t)b->n_voices;
        if (nv <= 32u)
            CUDA_TRY(s2::launch_ts_mix_rows(d_voice_out, nv, row_stride, (uint32_t)frames, d_bus_out, b->stream));
        else
            CUDA_TRY(s2::launch_bus_reduce(d_voice_out, nv, row_stride, (uint32_t)frames, d_bus_out, b->stream));
        g_launches.fetch_add(1, std::memory_order_relaxed);
    } else if (d_buses) {
        // per bus, the same rule over the bus's voice rows in voice order
        const Routes& R = b->route;
        s2::BusGroup g{};
        g.frames = (uint32_t)frames;
        g.buses = d_buses;
        g.bus_stride = bus_stride;
        g.rows = d_voice_out;
        g.row_stride = row_stride;
        g.idx = R.d + R.voices;
        g.spans = R.spans(R.ts_narrow);
        g.n_spans = R.n_ts_narrow;
        if (g.n_spans) CUDA_TRY(s2::launch_mix_rows_grouped(g, b->stream));
        g.spans = R.spans(R.ts_wide);
        g.n_spans = R.n_ts_wide;
        if (g.n_spans) CUDA_TRY(s2::launch_bus_reduce_grouped(g, b->stream));
        g_launches.fetch_add((R.n_ts_narrow ? 1 : 0) + (R.n_ts_wide ? 1 : 0), std::memory_order_relaxed);
    }
    ts.step++;
    ts.blocks++;
    b->total_frames += frames;
    b->max_offset += frames;
    return S2_OK;
}

// d_buses (routed banks only): every bus, bus g at d_buses + g * bus_stride, instead of the one bus d_bus_out.
int bank_render_impl(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_bus_out,
                     int trace, double* d_sum_sq = nullptr, uint32_t* d_peak = nullptr, float* d_buses = nullptr,
                     size_t bus_stride = 0) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (frames == 0) return S2_OK;
    if (frames > 0x7FFFFFFFull) return fail(S2_ERR_INVALID, "frames %zu too large for one call", frames);
    if (d_voice_out) {
        if (((uintptr_t)d_voice_out & 15u) != 0 || (row_stride & 3u) != 0 || row_stride < frames)
            return fail(S2_ERR_INVALID, "voice_out must be 16-byte aligned with row_stride %% 4 == 0 and >= frames");
    }
    if (b->max_offset + frames > 0xFFFFFFFFull) {
        // max_offset is an upper bound that only grows with the frames rendered; voices restarted since then sit at
        // small offsets.  Look at the real ones before failing (the reference panics only when a voice's own offset
        // overflows, process.rs:36): O(V), and only when the bound trips.
        uint64_t mx = 0;
        for (size_t i = 0; i < b->n_voices; i++)
            if (b->book[i].active) mx = std::max<uint64_t>(mx, (uint64_t)b->book[i].start_offset + (b->total_frames - b->book[i].start_total));
        b->max_offset = mx;
        if (mx + frames > 0xFFFFFFFFull) return fail(S2_ERR_OVERFLOW, "frame offset overflow (process.rs:36)");
    }
    CUDA_TRY(cudaSetDevice(b->device));
    if (trace == s2::TRACE_NONE) {
        const int cls = ts_block_class(b, frames, d_voice_out, d_sum_sq != nullptr);
        if (cls) return bank_render_time_split(b, frames, d_voice_out, row_stride, d_bus_out, cls == 2, d_buses, bus_stride);
    }
    b->split.main_dirty = true;   // the general kernels below move the carried phase on the bank's stream
    if (b->n_sub > 1 && trace == s2::TRACE_NONE)
        return bank_render_pipelined(b, frames, d_voice_out, row_stride, d_bus_out, d_sum_sq, d_peak, d_buses, bus_stride);
    if (b->n_sub > 1) {   // a trace: it renders the whole bank on the bank's stream
        int rc = settle_edits(b);
        if (rc) return rc;
    }

    const uint32_t n_warps = s2::render_warps((uint32_t)b->n_slots);
    s2::RenderArgs a = base_args(b, frames, d_voice_out, row_stride, d_sum_sq, d_peak);
    if (d_buses) {
        int rc = grow(b, &b->d_partials, 1, b->partials_cap, route_floats(b, frames));
        if (rc) return rc;
        route_args(b, a, b->d_partials);
    } else if (d_bus_out && bus_from_rows(b)) {
        int rc = grow(b, &b->d_partials, 1, b->partials_cap, b->n_voices * scratch_row_stride(frames));
        if (rc) return rc;
        rows_for_bus(a, b->d_partials, frames);
    } else if (d_bus_out) {
        if (n_warps == 1) {
            a.bus_partials = d_bus_out;   // a single warp sums its voices in index order: that IS the bus
        } else {
            int rc = grow(b, &b->d_partials, 1, b->partials_cap, partials_floats(n_warps, frames));
            if (rc) return rc;
            a.bus_partials = b->d_partials;
        }
    }
    CUDA_TRY(s2::launch_render(a, b->filter_kind, trace, b->stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    // the next pipelined render launches on the sub-streams, which do not wait for the bank's stream
    if (b->n_sub > 1) CUDA_TRY(cudaStreamSynchronize(b->stream));
    if (d_bus_out || d_buses) {
        int rc = d_buses ? route_mix(b, a, frames, d_buses, bus_stride, b->stream)
                 : bus_from_rows(b) ? mix_rows(b, a, frames, d_bus_out, b->stream)
                                    : mix_partials(b, a.bus_partials, n_warps, frames, d_bus_out, b->stream);
        if (rc) return rc;
    }
    b->total_frames += frames;
    b->max_offset += frames;
    return S2_OK;
}

// The order of one filter kind's voices `ids` (ascending voice indices) in their slots.  Groups of up to 32 voices
// keep the voice order, which for a bank of one kind keeps the bus sum in the reference's voice order.
void order_kind_group(const s2_voice_desc* voices, std::vector<uint32_t>& ids) {
    const size_t n = ids.size();
    if (n <= 32) return;
    // (inactive last) x oscillator kind x when the amp envelope comes to rest: the 32 voices of a warp then leave
    // the envelope ramps together instead of waiting for the slowest of a random draw.  Stable: a patch sweep
    // keeps the variants of one cutoff trajectory next to each other.
    // NOT a key: whether the cutoff follows the mod envelope.  Grouping the followers halves the warps that run
    // moving-cutoff chunks, but a step is one launch per voice range and a range's launches run in order: the
    // ranges of followers (1.9x the work per frame for 200 ms) fall behind the others and finish alone on a
    // part-filled machine.  Measured on the bench bank, first 20 blocks: 6.2 ms grouped and contiguous, 7.1 ms
    // grouped and dealt over the ranges, against mixed warps (every warp pays, all ranges in step).
    struct Key { uint32_t kind; float amp_rest; };
    auto key = [&](uint32_t v) -> Key {
        const s2_voice_desc& d = voices[v];
        return {d.active ? d.osc_kind : 4u, d.amp_attack_ms + d.amp_decay_ms};
    };
    std::stable_sort(ids.begin(), ids.end(), [&](uint32_t x, uint32_t y) {
        const Key a = key(x);
        const Key c = key(y);
        if (a.kind != c.kind) return a.kind < c.kind;
        return a.amp_rest < c.amp_rest;
    });
    // Instead the followers are PAIRED with voices whose cutoff rests: inside each kind, walking the sorted
    // order, a follower and a non-follower that are next in line share an aligned lane pair (2i, 2i + 1), and the
    // resting lane computes half of its partner's moving coefficients (chunk_modcut_pr).  Voices left without
    // a partner come after the pairs, in the sorted order.
    auto follows = [&](uint32_t v) { return voices[v].active && voices[v].mod_env_to_lpf_freq != 0.0f; };
    std::vector<uint32_t> out, fq, nq;
    out.reserve(n);
    size_t g0 = 0;
    while (g0 < n) {
        size_t g1 = g0;
        while (g1 < n && key(ids[g1]).kind == key(ids[g0]).kind) g1++;
        fq.clear(); nq.clear();
        size_t fi = 0, ni = 0;             // queue heads
        for (size_t i = g0; i < g1; i++) {
            const uint32_t v = ids[i];
            (follows(v) ? fq : nq).push_back(v);
            if (fi < fq.size() && ni < nq.size()) {
                if (out.size() & 1u) { out.push_back(nq[ni++]); continue; }    // keep the pairs on even slots
                out.push_back(fq[fi++]);
                out.push_back(nq[ni++]);
            }
        }
        // the unpaired: merge the two leftovers back into the sorted order
        std::vector<uint32_t> left(fq.begin() + fi, fq.end());
        left.insert(left.end(), nq.begin() + ni, nq.end());
        std::stable_sort(left.begin(), left.end(), [&](uint32_t x, uint32_t y) { return key(x).amp_rest < key(y).amp_rest; });
        out.insert(out.end(), left.begin(), left.end());
        g0 = g1;
    }
    ids.swap(out);
}

// The order in which `full_warps` sorted warps (32 slots each) are laid out: dealt round-robin into 8 bins laid out one
// after the other, so that every contiguous eighth / quarter / half of the slot range — the voice ranges of
// s2_bank_set_pipeline — holds the same mix of kinds and envelope lengths, and the ranges' streams advance together.
std::vector<size_t> deal_warps(size_t full_warps) {
    std::vector<size_t> order;
    order.reserve(full_warps);
    if (full_warps < 16) {
        for (size_t w = 0; w < full_warps; w++) order.push_back(w);
        return order;
    }
    for (size_t bin = 0; bin < 8; bin++)
        for (size_t w = bin; w < full_warps; w += 8) order.push_back(w);
    return order;
}

// The bank's slots: voice_of_slot, with kPadRow for a padding slot.  Voices are grouped by filter kind (stably, in
// kind order), each group is ordered by order_kind_group, and every group but the last is padded to whole warps of 32
// slots, so that each warp runs one filter.  With one kind there is no padding.
std::vector<uint32_t> layout_slots(const s2_voice_desc* voices, const std::vector<uint32_t>& kinds) {
    std::vector<uint32_t> slots;
    slots.reserve(kinds.size());
    std::vector<uint32_t> ids;
    for (uint32_t k = S2_FILTER_ONE_POLE; k <= S2_FILTER_FIRST_ORDER_HP; k++) {
        ids.clear();
        for (size_t v = 0; v < kinds.size(); v++)
            if (kinds[v] == k) ids.push_back((uint32_t)v);
        if (ids.empty()) continue;
        while (slots.size() & 31u) slots.push_back(s2::kPadRow);
        order_kind_group(voices, ids);
        slots.insert(slots.end(), ids.begin(), ids.end());
    }
    const size_t full_warps = slots.size() / 32;
    std::vector<uint32_t> dealt;
    dealt.reserve(slots.size());
    for (size_t w : deal_warps(full_warps)) dealt.insert(dealt.end(), slots.begin() + w * 32, slots.begin() + (w + 1) * 32);
    dealt.insert(dealt.end(), slots.begin() + full_warps * 32, slots.end());
    return dealt;
}

// A routed bank's slots.  Each bus's voices are laid out by layout_slots as a bank of those voices alone, each bus but
// the last non-empty one is padded to whole warps, and all the warps are dealt over the voice ranges (deal_warps).
// warps_of_bus[g] lists bus g's warps in that standalone bank's order, which is the order its partial rows are added
// in.  Voices of a bus keep their relative order: voice j of the standalone bank is the bus's j-th voice.
std::vector<uint32_t> layout_routed(const s2_voice_desc* voices, const std::vector<uint32_t>& kinds,
                                    const std::vector<uint32_t>& bus_of_voice, uint32_t n_buses,
                                    std::vector<std::vector<uint32_t>>& voices_of_bus,
                                    std::vector<std::vector<uint32_t>>& warps_of_bus) {
    voices_of_bus.assign(n_buses, {});
    for (size_t v = 0; v < kinds.size(); v++) voices_of_bus[bus_of_voice[v]].push_back((uint32_t)v);
    uint32_t last = 0;
    for (uint32_t g = 0; g < n_buses; g++)
        if (!voices_of_bus[g].empty()) last = g;
    std::vector<uint32_t> cat;                   // the buses' slots one after the other
    std::vector<uint32_t> owner;                 // bus of each warp of cat
    std::vector<s2_voice_desc> vg;
    std::vector<uint32_t> kg;
    for (uint32_t g = 0; g < n_buses; g++) {
        const std::vector<uint32_t>& ids = voices_of_bus[g];
        if (ids.empty()) continue;
        vg.clear(); kg.clear();
        for (uint32_t v : ids) { vg.push_back(voices[v]); kg.push_back(kinds[v]); }
        for (uint32_t s : layout_slots(vg.data(), kg)) cat.push_back(s == s2::kPadRow ? s : ids[s]);
        if (g != last) while (cat.size() & 31u) cat.push_back(s2::kPadRow);
        while (owner.size() * 32 < cat.size()) owner.push_back(g);
    }
    const size_t full_warps = cat.size() / 32;
    std::vector<size_t> order = deal_warps(full_warps);
    if (cat.size() & 31u) order.push_back(full_warps);
    std::vector<uint32_t> slots;
    slots.reserve(cat.size());
    warps_of_bus.assign(n_buses, {});
    std::vector<uint32_t> at(order.size());      // position of each warp of cat in the bank
    for (size_t i = 0; i < order.size(); i++) {
        at[order[i]] = (uint32_t)i;
        const size_t w0 = order[i] * 32;
        slots.insert(slots.end(), cat.begin() + w0, cat.begin() + std::min(w0 + 32, cat.size()));
    }
    for (size_t w = 0; w < order.size(); w++) warps_of_bus[owner[w]].push_back(at[w]);
    return slots;
}

// The device lists of a routed bank's bus reductions (Routes), and in scratch_index the bus-scratch row of every slot.
std::vector<uint32_t> route_words(Routes& R, const std::vector<std::vector<uint32_t>>& voices_of_bus,
                                  const std::vector<std::vector<uint32_t>>& warps_of_bus,
                                  const std::vector<uint32_t>& slot_of_voice, std::vector<uint32_t>& scratch_index) {
    const uint32_t n_buses = (uint32_t)voices_of_bus.size();
    std::vector<uint32_t> w, vstart(n_buses), wstart(n_buses), sstart(n_buses);
    std::vector<bool> from_rows(n_buses);
    R.voices = w.size();
    for (uint32_t g = 0; g < n_buses; g++) { vstart[g] = (uint32_t)(w.size() - R.voices); w.insert(w.end(), voices_of_bus[g].begin(), voices_of_bus[g].end()); }
    R.warps = w.size();
    for (uint32_t g = 0; g < n_buses; g++) { wstart[g] = (uint32_t)(w.size() - R.warps); w.insert(w.end(), warps_of_bus[g].begin(), warps_of_bus[g].end()); }
    // buses of up to 32 voices in several warps add their rows (bus_from_rows); their voices get bus-scratch rows
    for (uint32_t g = 0; g < n_buses; g++) {
        from_rows[g] = voices_of_bus[g].size() <= 32 && warps_of_bus[g].size() > 1;
        if (!from_rows[g]) continue;
        sstart[g] = R.n_scratch;
        for (uint32_t v : voices_of_bus[g]) scratch_index[slot_of_voice[v]] = R.n_scratch++;
    }
    R.iota = w.size();
    for (uint32_t i = 0; i < R.n_scratch; i++) w.push_back(i);
    auto span = [&](uint32_t g, uint32_t begin, size_t count) { w.push_back(g); w.push_back(begin); w.push_back((uint32_t)count); };
    R.rows_voice = w.size();
    for (uint32_t g = 0; g < n_buses; g++) if (from_rows[g]) { span(g, vstart[g], voices_of_bus[g].size()); R.n_rows++; }
    R.rows_scratch = w.size();
    for (uint32_t g = 0; g < n_buses; g++) if (from_rows[g]) span(g, sstart[g], voices_of_bus[g].size());
    R.partial = w.size();
    for (int big = 0; big < 2; big++)
        for (uint32_t g = 0; g < n_buses; g++) {
            if (from_rows[g] || (warps_of_bus[g].size() >= 512) != (big == 1)) continue;
            span(g, wstart[g], warps_of_bus[g].size());
            (big ? R.n_big : R.n_rest)++;
        }
    // time-split blocks: the rows of every bus, in voice order (launch_ts_mix_rows up to 32 voices, else the reduction)
    R.ts_narrow = w.size();
    for (uint32_t g = 0; g < n_buses; g++) if (voices_of_bus[g].size() <= 32) { span(g, vstart[g], voices_of_bus[g].size()); R.n_ts_narrow++; }
    R.ts_wide = w.size();
    for (uint32_t g = 0; g < n_buses; g++) if (voices_of_bus[g].size() > 32) { span(g, vstart[g], voices_of_bus[g].size()); R.n_ts_wide++; }
    return w;
}

// s2_bank_create, s2_bank_create_mixed and s2_bank_create_routed once their arguments are checked: `kinds` holds one
// valid filter kind per voice, and `bus_of_voice` one bus below n_buses per voice (or nothing: one bus).  Nothing is
// allocated on the device before every voice has passed validation.
int bank_create(int device, uint32_t sample_rate, std::vector<uint32_t> kinds, const s2_voice_desc* voices,
                void* stream, s2_bank** out, std::vector<uint32_t> bus_of_voice = {}, uint32_t n_buses = 1) {
    const size_t n_voices = kinds.size();
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(S2_ERR_NO_DEVICE, "no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(S2_ERR_NO_DEVICE, "device %d out of range (%d)", device, ndev);
    for (size_t i = 0; i < n_voices; i++) {
        int rc = validate_voice(voices[i], i, kinds[i]);
        if (rc) return rc;
    }
    std::vector<std::vector<uint32_t>> voices_of_bus, warps_of_bus;
    std::vector<uint32_t> voice_of_slot = n_buses > 1
        ? layout_routed(voices, kinds, bus_of_voice, n_buses, voices_of_bus, warps_of_bus) : layout_slots(voices, kinds);
    if (voice_of_slot.size() > 0x7FFFFFE0ull) return fail(S2_ERR_INVALID, "too many voices");
    CUDA_TRY(cudaSetDevice(device));

    s2_bank* b = new (std::nothrow) s2_bank;
    if (!b) return fail(S2_ERR_NOMEM, "out of host memory");
    b->device = device;
    b->stream = (cudaStream_t)stream;
    b->sample_rate = sample_rate;
    b->filter_kind = kinds[0];
    b->n_voices = n_voices;
    b->n_slots = voice_of_slot.size();
    b->vpad = (b->n_slots + 63) & ~(size_t)63;
    b->book.resize(n_voices);
    if (n_voices <= kTsMaxVoices) b->split.descs.assign(voices, voices + n_voices);
    if (const char* f = getenv("S2_FORCE_PATH")) b->force_path = (f[0] >= '1' && f[0] <= '3') ? (uint32_t)(f[0] - '0') : 0u;   // test hook

    b->voice_of_slot.swap(voice_of_slot);
    b->slot_of_voice.resize(n_voices);
    for (size_t s = 0; s < b->n_slots; s++) {
        const uint32_t v = b->voice_of_slot[s];
        if (v != s) b->identity = false;
        if (v != s2::kPadRow) b->slot_of_voice[v] = (uint32_t)s;
    }
    // The warp table: the plain one, and for a routed bank with buses added from their rows the one with
    // kWarpBusRows, followed by the bus-scratch row of every slot (s2_internal.h).
    const size_t n_warps = (b->n_slots + 31) / 32, wtb = s2::warp_table_bytes((uint32_t)b->vpad);
    std::vector<uint32_t> route, scratch_index(n_buses > 1 ? b->n_slots : 0, s2::kPadRow);
    if (n_buses > 1) route = route_words(b->route, voices_of_bus, warps_of_bus, b->slot_of_voice, scratch_index);
    std::vector<uint8_t> warp_kinds(b->route.n_scratch ? 2 * wtb + b->n_slots * sizeof(uint32_t) : n_warps);
    for (size_t w = 0; w < n_warps; w++) {
        const uint32_t v = b->voice_of_slot[w * 32];   // never padding
        const size_t bus_voices = n_buses > 1 ? voices_of_bus[bus_of_voice[v]].size() : n_voices;
        warp_kinds[w] = (uint8_t)(kinds[v] | (bus_voices <= 32 ? s2::kWarpNarrowBus : 0u));
        if (b->route.n_scratch)
            warp_kinds[wtb + w] = warp_kinds[w] | (scratch_index[b->slot_of_voice[v]] != s2::kPadRow ? s2::kWarpBusRows : 0u);
    }
    if (b->route.n_scratch) memcpy(warp_kinds.data() + 2 * wtb, scratch_index.data(), b->n_slots * sizeof(uint32_t));
    uint32_t seen = 0;
    for (uint32_t k : kinds) seen |= 1u << k;
    b->n_kinds = (uint32_t)__builtin_popcount(seen);
    b->voice_kind.swap(kinds);
    b->n_buses = n_buses;
    if (n_buses > 1) b->bus_of_voice.swap(bus_of_voice);
    // every routed bank renders through the per-warp kernel, which reads each warp's bus width from the table
    const bool warp_table = b->n_kinds > 1 || n_buses > 1;
    const size_t counters = std::max<size_t>(1, b->route.n_big) * s2::kBusCounters;

    std::vector<float> hp((size_t)s2::P_COUNT * b->vpad, 0.0f), hs((size_t)s2::S_COUNT * b->vpad, 0.0f);
    for (size_t s = 0; s < b->n_slots; s++)
        if (b->voice_of_slot[s] == s2::kPadRow) hp[(size_t)s2::P_ROW * b->vpad + s] = ubits(s2::kPadRow);   // inactive: zeros
    for (size_t i = 0; i < n_voices; i++) {
        const size_t slot = b->slot_of_voice[i];
        pack_voice(voices[i], (uint32_t)i, hp.data() + slot, b->vpad);
        s2_voice_state st;
        memset(&st, 0, sizeof st);
        st.frame_offset = voices[i].frame_offset;
        pack_state(st, hs.data() + slot, b->vpad);
        b->book[i] = {voices[i].frame_offset, 0, voices[i].active ? 1u : 0u, voices[i].osc_kind};
        if (voices[i].active && voices[i].frame_offset > b->max_offset) b->max_offset = voices[i].frame_offset;
        if (voices[i].osc_kind == S2_OSC_SINE) b->n_sine++;
    }
    cudaError_t e = cudaMalloc(&b->d_params, hp.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_state, hs.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc(&b->d_bus_counters, counters * sizeof(unsigned int));
    if (e == cudaSuccess) e = cudaMemsetAsync(b->d_bus_counters, 0, counters * sizeof(unsigned int), b->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_params, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->d_state, hs.data(), hs.size() * sizeof(float), cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess && warp_table) e = cudaMalloc(&b->d_warp_kinds, warp_kinds.size());
    if (e == cudaSuccess && warp_table)
        e = cudaMemcpyAsync(b->d_warp_kinds, warp_kinds.data(), warp_kinds.size(), cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess && !route.empty()) e = cudaMalloc(&b->route.d, route.size() * sizeof(uint32_t));
    if (e == cudaSuccess && !route.empty())
        e = cudaMemcpyAsync(b->route.d, route.data(), route.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
    if (e != cudaSuccess) {
        int rc = fail(e == cudaErrorMemoryAllocation ? S2_ERR_NOMEM : S2_ERR_CUDA, "bank upload: %s", cudaGetErrorString(e));
        s2_bank_destroy(b);
        return rc;
    }
    *out = b;
    return S2_OK;
}

}  // namespace

extern "C" {

uint32_t s2_abi_version(void) { return S2_ABI_VERSION; }
const char* s2_last_error(void) { return g_err; }
uint64_t s2_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int s2_device_count(int* count) {
    if (!count) return fail(S2_ERR_INVALID, "null count");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(S2_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count = n;
    return S2_OK;
}

// synth.rs:208-212
float s2_note_to_pitch(uint8_t note) {
    const float n = (float)note;
    return 440.0f * powf(2.0f, (n - 69.0f) / 12.0f);
}

// synth.rs:125-152
void s2_default_voice(s2_voice_desc* d) {
    if (!d) return;
    memset(d, 0, sizeof *d);
    d->osc_kind = S2_OSC_SAW;
    d->noise_seed = 0;
    d->pitch_hz = 440.0f;
    d->osc_gain = 1.0f;
    d->noise_amt = 0.0f;
    d->lpf_freq_hz = 200.0f;
    d->damping = 1.41421356f;
    d->amp_attack_ms = 100.0f; d->amp_decay_ms = 100.0f; d->amp_sustain = 0.5f; d->amp_release_ms = 100.0f;
    d->mod_attack_ms = 0.0f; d->mod_decay_ms = 200.0f; d->mod_sustain = 0.0f; d->mod_release_ms = 0.0f;
    d->mod_env_to_osc_freq = 0.0f;
    d->mod_env_to_lpf_freq = 10.0f;
    d->frame_offset = 0;
    d->release_offset = S2_NO_RELEASE;
    d->active = 0;
}

int s2_bank_create(int device, uint32_t sample_rate, uint32_t filter_kind, size_t n_voices,
                   const s2_voice_desc* voices, void* stream, s2_bank** out) {
    if (!out) return fail(S2_ERR_INVALID, "null out");
    *out = nullptr;
    if (n_voices == 0 || !voices) return fail(S2_ERR_INVALID, "empty bank");
    if (n_voices > 0x7FFFFFE0ull) return fail(S2_ERR_INVALID, "too many voices");
    if (sample_rate == 0) return fail(S2_ERR_INVALID, "sample_rate must be > 0");
    if (filter_kind > S2_FILTER_FIRST_ORDER_HP) return fail(S2_ERR_INVALID, "filter_kind %u", filter_kind);
    return bank_create(device, sample_rate, std::vector<uint32_t>(n_voices, filter_kind), voices, stream, out);
}

int s2_bank_create_mixed(int device, uint32_t sample_rate, size_t n_voices, const s2_voice_desc* voices,
                         const uint32_t* filter_kinds, void* stream, s2_bank** out) {
    if (!out) return fail(S2_ERR_INVALID, "null out");
    *out = nullptr;
    if (n_voices == 0 || !voices) return fail(S2_ERR_INVALID, "empty bank");
    if (!filter_kinds) return fail(S2_ERR_INVALID, "null filter_kinds");
    if (n_voices > 0x7FFFFFE0ull) return fail(S2_ERR_INVALID, "too many voices");
    if (sample_rate == 0) return fail(S2_ERR_INVALID, "sample_rate must be > 0");
    for (size_t i = 0; i < n_voices; i++)
        if (filter_kinds[i] > S2_FILTER_FIRST_ORDER_HP)
            return fail(S2_ERR_INVALID, "voice %zu: filter_kind %u", i, filter_kinds[i]);
    return bank_create(device, sample_rate, std::vector<uint32_t>(filter_kinds, filter_kinds + n_voices), voices,
                       stream, out);
}

int s2_bank_create_routed(int device, uint32_t sample_rate, size_t n_voices, const s2_voice_desc* voices,
                          const uint32_t* filter_kinds, const uint32_t* bus_of_voice, uint32_t n_buses,
                          void* stream, s2_bank** out) {
    if (!out) return fail(S2_ERR_INVALID, "null out");
    *out = nullptr;
    if (n_voices == 0 || !voices) return fail(S2_ERR_INVALID, "empty bank");
    if (!filter_kinds) return fail(S2_ERR_INVALID, "null filter_kinds");
    if (!bus_of_voice) return fail(S2_ERR_INVALID, "null bus_of_voice");
    if (n_buses == 0 || n_buses > S2_MAX_BUSES) return fail(S2_ERR_INVALID, "n_buses must be in [1, %u]", S2_MAX_BUSES);
    if (n_voices > 0x7FFFFFE0ull) return fail(S2_ERR_INVALID, "too many voices");
    if (sample_rate == 0) return fail(S2_ERR_INVALID, "sample_rate must be > 0");
    for (size_t i = 0; i < n_voices; i++) {
        if (filter_kinds[i] > S2_FILTER_FIRST_ORDER_HP)
            return fail(S2_ERR_INVALID, "voice %zu: filter_kind %u", i, filter_kinds[i]);
        if (bus_of_voice[i] >= n_buses) return fail(S2_ERR_INVALID, "voice %zu: bus %u of %u", i, bus_of_voice[i], n_buses);
    }
    std::vector<uint32_t> kinds(filter_kinds, filter_kinds + n_voices);
    if (n_buses == 1) return bank_create(device, sample_rate, std::move(kinds), voices, stream, out);   // a mixed bank
    return bank_create(device, sample_rate, std::move(kinds), voices, stream, out,
                       std::vector<uint32_t>(bus_of_voice, bus_of_voice + n_voices), n_buses);
}

void s2_bank_destroy(s2_bank* b) {
    if (!b) return;
    cudaSetDevice(b->device);
    bank_drain(b);
    cudaStreamSynchronize(b->stream);
    b->pipe.release();
    b->split.release();
    b->batches.release();
    cudaFree(b->d_params);
    cudaFree(b->d_state);
    cudaFree(b->d_partials);
    cudaFree(b->d_bus_counters);
    cudaFree(b->d_bus);
    cudaFree(b->d_warp_kinds);
    cudaFree(b->route.d);
    delete b;
}

size_t s2_bank_voices(const s2_bank* b) { return b ? b->n_voices : 0; }

int s2_bank_filter_kinds(const s2_bank* b, uint32_t* out) {
    if (!b || !out) return fail(S2_ERR_INVALID, "null argument");
    std::copy(b->voice_kind.begin(), b->voice_kind.end(), out);
    return S2_OK;
}

int s2_bank_buses(const s2_bank* b, uint32_t* n_buses, uint32_t* bus_of_voice) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (n_buses) *n_buses = b->n_buses;
    if (bus_of_voice) {
        if (b->bus_of_voice.empty()) std::fill(bus_of_voice, bus_of_voice + b->n_voices, 0u);
        else std::copy(b->bus_of_voice.begin(), b->bus_of_voice.end(), bus_of_voice);
    }
    return S2_OK;
}

int s2_bank_set_voice(s2_bank* b, size_t index, const s2_voice_desc* voice) {
    if (!b || !voice) return fail(S2_ERR_INVALID, "null argument");
    if (index >= b->n_voices) return fail(S2_ERR_INVALID, "voice index %zu out of range", index);
    int rc = validate_voice(*voice, index, b->voice_kind[index]);
    if (rc) return rc;
    CUDA_TRY(cudaSetDevice(b->device));
    if ((rc = settle_edits(b)) != S2_OK) return rc;    // pipelined mode: per-voice edits are not pipelined
    float hp[s2::P_COUNT], hs[s2::S_COUNT];
    const size_t slot = b->slot_of_voice[index];   // the voice keeps its slot (a changed kind makes that warp mixed)
    pack_note_on(*voice, (uint32_t)index, hp, hs, 1);
    // one 4-byte element per SoA row
    CUDA_TRY(cudaMemcpy2DAsync(b->d_params + slot, b->vpad * sizeof(float), hp, sizeof(float), sizeof(float),
                               s2::P_COUNT, cudaMemcpyHostToDevice, b->stream));
    CUDA_TRY(cudaMemcpy2DAsync(b->d_state + slot, b->vpad * sizeof(float), hs, sizeof(float), sizeof(float),
                               s2::S_COUNT, cudaMemcpyHostToDevice, b->stream));
    CUDA_TRY(cudaStreamSynchronize(b->stream));   // hp/hs live on this stack frame
    note_voice(b, index, *voice);
    return S2_OK;
}

int s2_bank_set_voices(s2_bank* b, size_t n, const uint32_t* indices, const s2_voice_desc* voices) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (n == 0) return S2_OK;
    if (!indices || !voices) return fail(S2_ERR_INVALID, "null argument");
    for (size_t j = 0; j < n; j++) {
        if (indices[j] >= b->n_voices) return fail(S2_ERR_INVALID, "entry %zu: voice index %u out of range", j, indices[j]);
        int rc = validate_voice(voices[j], indices[j], b->voice_kind[indices[j]]);
        if (rc) return rc;
    }
    CUDA_TRY(cudaSetDevice(b->device));
    VoiceBatches& vb = b->batches;
    Pipeline& pl = b->pipe;
    { int rc = vb.create(); if (rc) return rc; }

    // The last entry of each index wins: walking backwards, an index is kept the first time it is met.  The kept
    // entries are then bucketed by voice range (one range unless pipelined), each bucket contiguous in the batch.
    if (vb.stamp.size() != b->n_voices) vb.stamp.assign(b->n_voices, 0u);
    if (++vb.gen == 0) { std::fill(vb.stamp.begin(), vb.stamp.end(), 0u); vb.gen = 1; }
    const int n_ranges = b->n_sub;
    uint32_t bound[9];
    for (int k = 0; k <= n_ranges; k++) bound[k] = n_ranges > 1 ? sub_begin(b, k) : (k ? (uint32_t)b->n_slots : 0u);
    std::vector<uint32_t> kept;
    std::vector<uint8_t> range_of;
    size_t count[8] = {}, begin[8] = {};
    for (size_t j = n; j-- > 0;) {
        if (vb.stamp[indices[j]] == vb.gen) continue;
        vb.stamp[indices[j]] = vb.gen;
        const uint32_t slot = b->slot_of_voice[indices[j]];
        int k = 0;
        while (slot >= bound[k + 1]) k++;
        kept.push_back((uint32_t)j);
        range_of.push_back((uint8_t)k);
        count[k]++;
    }
    for (int k = 1; k < n_ranges; k++) begin[k] = begin[k - 1] + count[k - 1];
    const size_t m = kept.size();
    const size_t need = (size_t)(s2::P_COUNT + s2::S_COUNT + 1) * m;

    const int r = (int)(vb.next % (uint64_t)kBatchBufs);
    if (need > vb.h_cap) {
        for (int i = 0; i < kBatchBufs; i++) CUDA_TRY(cudaEventSynchronize(vb.ev_copied[i]));   // no copy reads them
        int rc = grow(b, vb.h, kBatchBufs, vb.h_cap, need, true);
        if (rc) return rc;
    }
    { int rc = grow(b, vb.d, kBatchBufs, vb.d_cap, need); if (rc) return rc; }
    CUDA_TRY(cudaEventSynchronize(vb.ev_copied[r]));   // h[r] is free again (long since, in steady state)
    float* hb = vb.h[r];
    size_t fill[8];
    std::copy(begin, begin + 8, fill);
    for (size_t i = 0; i < m; i++) {
        const uint32_t j = kept[i];
        const size_t e = fill[range_of[i]]++;
        pack_note_on(voices[j], indices[j], hb + e, hb + (size_t)s2::P_COUNT * m + e, m);
        hb[(size_t)(s2::P_COUNT + s2::S_COUNT) * m + e] = ubits(b->slot_of_voice[indices[j]]);
    }

    if (n_ranges == 1) {
        // one stream (time-split included): copy and scatter in order on the bank's stream
        CUDA_TRY(cudaMemcpyAsync(vb.d[r], hb, need * sizeof(float), cudaMemcpyHostToDevice, b->stream));
        CUDA_TRY(cudaEventRecord(vb.ev_copied[r], b->stream));
        CUDA_TRY(s2::launch_set_voices(vb.d[r], (uint32_t)m, 0, (uint32_t)m, b->d_params, b->d_state, (uint32_t)b->vpad,
                                       nullptr, b->stream));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        b->split.main_dirty = true;   // the next phase pre-pass reads the fresh phases
    } else {
        // Pipelined: the copy on the upload stream, then each range that has entries scatters them on its own
        // stream, between its renders.  No range waits for another.  A pending note-off table is applied by the
        // ranges' next renders: the scatter writes the note-ons' release offsets into it too (after it has landed).
        for (int k = 0; k < n_ranges; k++) CUDA_TRY(cudaStreamWaitEvent(pl.upload, vb.ev_read[r][k], 0));   // d[r] free
        CUDA_TRY(cudaMemcpyAsync(vb.d[r], hb, need * sizeof(float), cudaMemcpyHostToDevice, pl.upload));
        CUDA_TRY(cudaEventRecord(vb.ev_copied[r], pl.upload));
        const int q = pl.table_pending;
        for (int k = 0; k < n_ranges; k++) {
            if (!count[k]) continue;
            cudaStream_t sk = pl.sub[k];
            CUDA_TRY(cudaStreamWaitEvent(sk, vb.ev_copied[r], 0));
            if (q >= 0) CUDA_TRY(cudaStreamWaitEvent(sk, pl.ev_stage[q], 0));
            CUDA_TRY(s2::launch_set_voices(vb.d[r], (uint32_t)m, (uint32_t)begin[k], (uint32_t)count[k], b->d_params,
                                           b->d_state, (uint32_t)b->vpad, q >= 0 ? pl.d_staging[q] : nullptr, sk));
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CUDA_TRY(cudaEventRecord(vb.ev_read[r][k], sk));
            if (q >= 0) CUDA_TRY(cudaEventRecord(pl.ev_gather[k][q], sk));   // a superseding table waits for it
            CUDA_TRY(cudaEventRecord(pl.ev_sub[k], sk));
        }
    }
    vb.next++;
    for (size_t j = 0; j < n; j++) note_voice(b, indices[j], voices[j]);
    return S2_OK;
}

int s2_bank_release_voice(s2_bank* b, size_t index) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (index >= b->n_voices) return fail(S2_ERR_INVALID, "voice index %zu out of range", index);
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = settle_edits(b); if (rc) return rc; }
    const uint32_t rel = current_offset(b, index);   // release_frame_offset = current_frame_offset (synth.rs:75)
    CUDA_TRY(cudaMemcpyAsync(b->d_params + (size_t)s2::P_RELEASE * b->vpad + b->slot_of_voice[index], &rel,
                             sizeof rel, cudaMemcpyHostToDevice, b->stream));
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    if (!b->split.descs.empty()) b->split.descs[index].release_offset = rel;
    return S2_OK;
}

int s2_bank_set_releases(s2_bank* b, const uint32_t* h_release) {
    if (!b || !h_release) return fail(S2_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(b->device));
    for (size_t i = 0; i < b->split.descs.size(); i++) b->split.descs[i].release_offset = h_release[i];
    Pipeline& pl = b->pipe;
    if (b->n_sub > 1) {
        // stage the table on the mix stream; every sub-bank applies it to its own slots right before its
        // next render (bank_render_pipelined), so no sub-bank waits for another
        const int q = (int)(pl.table_step & 1u);
        if (pl.table_pending >= 0) {
            // two tables without a render in between: the older one is simply superseded
            pl.table_pending = -1;
            pl.table_step--;
            return s2_bank_set_releases(b, h_release);
        }
        // buffer q may still feed the renders that apply the table staged two uploads ago, or, when this table
        // supersedes one, the s2_bank_set_voices scatters that wrote into it
        for (int k = 0; k < b->n_sub; k++) CUDA_TRY(cudaStreamWaitEvent(pl.upload, pl.ev_gather[k][q], 0));
        CUDA_TRY(cudaMemcpyAsync(pl.d_staging[q], h_release, b->n_voices * sizeof(uint32_t), cudaMemcpyHostToDevice, pl.upload));
        CUDA_TRY(cudaEventRecord(pl.ev_stage[q], pl.upload));
        pl.table_pending = q;
        pl.table_step++;
        return S2_OK;
    }
    uint32_t* row = reinterpret_cast<uint32_t*>(b->d_params + (size_t)s2::P_RELEASE * b->vpad);
    if (b->identity) {
        CUDA_TRY(cudaMemcpyAsync(row, h_release, b->n_voices * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream));
        return S2_OK;
    }
    // Permuted slots on one stream: stage in voice order, gather into slot order.  Staging buffer 0 is free here:
    // s2_bank_set_pipeline synchronises every stream when the ranges change, and no table is pending while n_sub == 1.
    if (!pl.d_staging[0]) CUDA_TRY(cudaMalloc(&pl.d_staging[0], b->n_voices * sizeof(uint32_t)));
    CUDA_TRY(cudaMemcpyAsync(pl.d_staging[0], h_release, b->n_voices * sizeof(uint32_t), cudaMemcpyHostToDevice, b->stream));
    CUDA_TRY(s2::launch_gather_u32(pl.d_staging[0], b->d_params + (size_t)s2::P_ROW * b->vpad, row,
                                   (uint32_t)b->n_slots, b->stream));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return S2_OK;
}

int s2_bank_render(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_bus_out) {
    return bank_render_impl(b, frames, d_voice_out, row_stride, d_bus_out, s2::TRACE_NONE);
}

int s2_bank_render_metered(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_bus_out,
                           double* d_sum_sq, float* d_peak) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (!d_sum_sq || !d_peak) return fail(S2_ERR_INVALID, "null meter (sum_sq and peak are both required)");
    if (((uintptr_t)d_sum_sq & 7u) != 0 || ((uintptr_t)d_peak & 3u) != 0)
        return fail(S2_ERR_INVALID, "sum_sq must be 8-byte and peak 4-byte aligned");
    return bank_render_impl(b, frames, d_voice_out, row_stride, d_bus_out, s2::TRACE_NONE, d_sum_sq,
                            reinterpret_cast<uint32_t*>(d_peak));
}

int s2_bank_render_buses(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* d_buses,
                         size_t bus_stride, double* d_sum_sq, float* d_peak) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (!d_buses) return fail(S2_ERR_INVALID, "null d_buses");
    if (((uintptr_t)d_buses & 15u) != 0 || (bus_stride & 3u) != 0 || bus_stride < frames)
        return fail(S2_ERR_INVALID, "d_buses must be 16-byte aligned with bus_stride %% 4 == 0 and >= frames");
    if (!d_sum_sq != !d_peak) return fail(S2_ERR_INVALID, "null meter (sum_sq and peak are given together)");
    if (((uintptr_t)d_sum_sq & 7u) != 0 || ((uintptr_t)d_peak & 3u) != 0)
        return fail(S2_ERR_INVALID, "sum_sq must be 8-byte and peak 4-byte aligned");
    uint32_t* peak = reinterpret_cast<uint32_t*>(d_peak);
    if (b->n_buses == 1)   // one bus: the bank's mono bus
        return bank_render_impl(b, frames, d_voice_out, row_stride, d_buses, s2::TRACE_NONE, d_sum_sq, peak);
    return bank_render_impl(b, frames, d_voice_out, row_stride, nullptr, s2::TRACE_NONE, d_sum_sq, peak, d_buses,
                            bus_stride);
}

int s2_bank_trace_phase(s2_bank* b, size_t frames, float* d_phase_out, size_t row_stride) {
    if (!d_phase_out) return fail(S2_ERR_INVALID, "null phase_out");
    return bank_render_impl(b, frames, d_phase_out, row_stride, nullptr, s2::TRACE_PHASE);
}

int s2_bank_render_bus_host(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* h_bus_out) {
    int rc = s2_bank_render_bus_host_async(b, frames, d_voice_out, row_stride, h_bus_out);
    if (rc) return rc;
    if (frames == 0) return S2_OK;
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    return S2_OK;
}

int s2_bank_render_bus_host_async(s2_bank* b, size_t frames, float* d_voice_out, size_t row_stride, float* h_bus_out) {
    if (!b || !h_bus_out) return fail(S2_ERR_INVALID, "null argument");
    if (frames == 0) return S2_OK;
    CUDA_TRY(cudaSetDevice(b->device));
    int rc = grow(b, &b->d_bus, 1, b->bus_cap, frames);
    if (rc) return rc;
    rc = bank_render_impl(b, frames, d_voice_out, row_stride, b->d_bus, s2::TRACE_NONE);
    if (rc) return rc;
    if (b->n_sub > 1) {
        // pipelined: the mix lives on the bank's mix stream; the caller's stream only waits for the copy
        CUDA_TRY(cudaMemcpyAsync(h_bus_out, b->d_bus, frames * sizeof(float), cudaMemcpyDeviceToHost, b->pipe.mix));
        CUDA_TRY(cudaEventRecord(b->pipe.ev_tail, b->pipe.mix));
        CUDA_TRY(cudaStreamWaitEvent(b->stream, b->pipe.ev_tail, 0));
        return S2_OK;
    }
    CUDA_TRY(cudaMemcpyAsync(h_bus_out, b->d_bus, frames * sizeof(float), cudaMemcpyDeviceToHost, b->stream));
    return S2_OK;
}

int s2_bank_get_state(s2_bank* b, s2_voice_state* out) {
    if (!b || !out) return fail(S2_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = bank_drain(b); if (rc) return rc; }
    std::vector<float> hs((size_t)s2::S_COUNT * b->vpad);
    CUDA_TRY(cudaMemcpyAsync(hs.data(), b->d_state, hs.size() * sizeof(float), cudaMemcpyDeviceToHost, b->stream));
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    const size_t p = b->vpad;
    for (size_t v = 0; v < b->n_voices; v++) {
        const size_t i = b->slot_of_voice[v];
        s2_voice_state& s = out[v];
        s.phase = hs[s2::S_PHASE * p + i];
        s.has_phase = fbits(hs[s2::S_HAS_PHASE * p + i]);
        s.frame_offset = fbits(hs[s2::S_OFFSET * p + i]);
        s.lpf_last = hs[s2::S_LAST * p + i];
        s.x1 = hs[s2::S_X1 * p + i];
        s.x2 = hs[s2::S_X2 * p + i];
        s.y1 = hs[s2::S_Y1 * p + i];
        s.y2 = hs[s2::S_Y2 * p + i];
    }
    return S2_OK;
}

int s2_bank_set_state(s2_bank* b, const s2_voice_state* in) {
    if (!b || !in) return fail(S2_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = bank_drain(b); if (rc) return rc; }
    std::vector<float> hs((size_t)s2::S_COUNT * b->vpad, 0.0f);
    uint64_t mx = 0;
    for (size_t i = 0; i < b->n_voices; i++) {
        pack_state(in[i], hs.data() + b->slot_of_voice[i], b->vpad);
        b->book[i].start_offset = in[i].frame_offset;
        b->book[i].start_total = b->total_frames;
        if (b->book[i].active && in[i].frame_offset > mx) mx = in[i].frame_offset;
    }
    b->max_offset = mx;
    CUDA_TRY(cudaMemcpyAsync(b->d_state, hs.data(), hs.size() * sizeof(float), cudaMemcpyHostToDevice, b->stream));
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    return S2_OK;
}

int s2_bank_sync(s2_bank* b) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = bank_drain(b); if (rc) return rc; }
    CUDA_TRY(cudaStreamSynchronize(b->stream));
    return S2_OK;
}

int s2_bank_set_pipeline(s2_bank* b, int n_sub) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (n_sub < 1 || n_sub > 8) return fail(S2_ERR_INVALID, "n_sub must be in [1, 8]");
    if (n_sub > 1 && b->split.enabled) return fail(S2_ERR_INVALID, "time-split and pipelined voice ranges are exclusive");
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = s2_bank_sync(b); if (rc == S2_OK) rc = settle_edits(b); if (rc) return rc; }
    if (n_sub > 1) { int rc = b->pipe.create(n_sub, b->n_voices); if (rc) return rc; }
    b->n_sub = n_sub;
    b->pipe.step = 0;
    b->pipe.table_step = 0;
    b->pipe.table_pending = -1;
    return S2_OK;
}

int s2_bank_set_time_split(s2_bank* b, int enable) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    CUDA_TRY(cudaSetDevice(b->device));
    { int rc = s2_bank_sync(b); if (rc) return rc; }
    if (!enable) { b->split.enabled = false; return S2_OK; }
    if (b->n_kinds > 1) return fail(S2_ERR_INVALID, "time-split rendering takes banks of one filter kind");
    if (b->filter_kind > S2_FILTER_BIQUAD_LP)
        return fail(S2_ERR_INVALID, "time-split rendering knows the one-pole and the second-order low-pass filters");
    if (b->n_voices > kTsMaxVoices)
        return fail(S2_ERR_INVALID, "time-split rendering is for narrow banks (<= %zu voices)", kTsMaxVoices);
    if (b->n_sub > 1) return fail(S2_ERR_INVALID, "time-split and pipelined voice ranges are exclusive");
    { int rc = b->split.create(b->n_slots); if (rc) return rc; }
    b->split.enabled = true;
    b->split.main_dirty = true;
    b->split.step = 0;
    return S2_OK;
}

int s2_bank_time_split_blocks(s2_bank* b, uint64_t* blocks) {
    if (!b || !blocks) return fail(S2_ERR_INVALID, "null argument");
    *blocks = b->split.blocks;
    return S2_OK;
}

int s2_bank_join(s2_bank* b, void* stream) {
    if (!b) return fail(S2_ERR_INVALID, "null bank");
    if (b->n_sub <= 1) return S2_OK;       // everything already is on the bank's stream
    CUDA_TRY(cudaSetDevice(b->device));
    cudaStream_t st = (cudaStream_t)stream;
    for (int k = 0; k < b->n_sub; k++) CUDA_TRY(cudaStreamWaitEvent(st, b->pipe.ev_sub[k], 0));
    CUDA_TRY(cudaEventRecord(b->pipe.ev_tail, b->pipe.mix));
    CUDA_TRY(cudaStreamWaitEvent(st, b->pipe.ev_tail, 0));
    return S2_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// Synth mirror (s2_lib/src/try3/synth.rs)

namespace {
constexpr int kNumVoices = 8;   // synth.rs:7

struct SynthVoice {             // synth.rs:23-30 (DSP state lives on the device)
    uint8_t note = 0;
    float velocity = 0.0f;      // stored, never read by the DSP (synth.rs:26)
    bool has_current = false;
    bool has_release = false;
    uint32_t release = 0;
};
}  // namespace

struct s2_synth {
    int device = 0;
    s2_bank* bank = nullptr;    // created by the first sample() call, which is when the rate is known
    uint32_t sample_rate = 0;
    SynthVoice voices[kNumVoices];
    // note events that arrived before the bank exists
    s2_voice_desc pending[kNumVoices];
    bool dirty[kNumVoices] = {};
    s2_patch patch;             // what note_on plays: Synth::default_config() unless s2_synth_set_patch changed it
    float* d_score = nullptr;   // device buffer of s2_synth_render_score
    size_t score_cap = 0;
};

namespace {

uint32_t synth_current(const s2_synth* s, int i) {
    if (!s->voices[i].has_current) return 0xFFFFFFFFu;   // unwrap_or(u32::MAX), synth.rs:106-107
    if (s->bank && !s->dirty[i]) return current_offset(s->bank, (size_t)i);
    return s->pending[i].frame_offset;
}

// The note-ons since the last render, as one batch on the bank's stream (no host wait).
int synth_flush(s2_synth* s) {
    uint32_t idx[kNumVoices];
    s2_voice_desc ds[kNumVoices];
    size_t n = 0;
    for (int i = 0; i < kNumVoices; i++)
        if (s->dirty[i]) { idx[n] = (uint32_t)i; ds[n++] = s->pending[i]; }
    int rc = s2_bank_set_voices(s->bank, n, idx, ds);
    if (rc) return rc;
    for (int i = 0; i < kNumVoices; i++) s->dirty[i] = false;
    return S2_OK;
}

}  // namespace

extern "C" {

int s2_synth_new(int device, s2_synth** out) {
    if (!out) return fail(S2_ERR_INVALID, "null out");
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(S2_ERR_NO_DEVICE, "no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return fail(S2_ERR_NO_DEVICE, "device %d out of range (%d)", device, ndev);
    s2_synth* s = new (std::nothrow) s2_synth;
    if (!s) return fail(S2_ERR_NOMEM, "out of host memory");
    s->device = device;
    for (int i = 0; i < kNumVoices; i++) s2_default_voice(&s->pending[i]);   // Voice::default(): free slot
    s2_default_patch(&s->patch);
    *out = s;
    return S2_OK;
}

void s2_synth_free(s2_synth* s) {
    if (!s) return;
    s2_bank_destroy(s->bank);
    if (s->d_score) cudaFree(s->d_score);
    delete s;
}

// synth.rs:61-70 + next_voice :101-120: the first slot with the strictly greatest offset; free = u32::MAX
int s2_synth_note_on(s2_synth* s, uint8_t note, float velocity) {
    if (!s) return fail(S2_ERR_INVALID, "null synth");
    int oldest = 0;
    for (int i = 1; i < kNumVoices; i++)
        if (synth_current(s, i) > synth_current(s, oldest)) oldest = i;
    SynthVoice& v = s->voices[oldest];
    v.note = note;
    v.velocity = velocity;
    v.has_current = true;
    v.has_release = false;
    v.release = 0;
    s2_voice_desc d = s->patch.voice;
    d.pitch_hz = s2_note_to_pitch(note);
    d.frame_offset = 0;
    d.release_offset = S2_NO_RELEASE;
    d.active = 1;
    s->pending[oldest] = d;
    s->dirty[oldest] = true;
    return S2_OK;
}

// synth.rs:72-99: the LAST active voice holding that note
int s2_synth_note_off(s2_synth* s, uint8_t note) {
    if (!s) return fail(S2_ERR_INVALID, "null synth");
    int found = -1;
    for (int i = 0; i < kNumVoices; i++) {
        const SynthVoice& v = s->voices[i];
        if (v.note == note && v.has_current && !v.has_release) found = i;
    }
    if (found < 0) return S2_OK;
    SynthVoice& v = s->voices[found];
    v.has_release = true;
    v.release = synth_current(s, found);
    s->pending[found].release_offset = v.release;      // the description mirrors the bank (rebuilds start from it)
    if (s->dirty[found] || !s->bank) {
        s->dirty[found] = true;
        return S2_OK;
    }
    return s2_bank_release_voice(s->bank, (size_t)found);
}

// The bank is created by the first render, which is when the rate is known (synth.rs:156 takes it per call).
static int synth_ensure_bank(s2_synth* s, uint32_t sample_rate) {
    if (s->bank && s->sample_rate != sample_rate) {
        // Changing the rate mid-stream re-derives every rate-dependent constant; carry the DSP state over
        // into a bank built for the new rate.
        std::vector<s2_voice_state> st(kNumVoices);
        std::vector<s2_voice_desc> ds(kNumVoices);
        int rc = s2_bank_get_state(s->bank, st.data());
        if (rc) return rc;
        for (int i = 0; i < kNumVoices; i++) {
            ds[i] = s->pending[i];
            if (!s->dirty[i]) ds[i].frame_offset = st[i].frame_offset;
            // a note_off on an uploaded voice went straight to the bank: the description must carry it too
            ds[i].release_offset = s->voices[i].has_release ? s->voices[i].release : S2_NO_RELEASE;
        }
        s2_bank* nb = nullptr;
        rc = s2_bank_create(s->device, sample_rate, s->patch.filter_kind, kNumVoices, ds.data(), nullptr, &nb);
        if (rc) return rc;
        for (int i = 0; i < kNumVoices; i++)
            if (s->dirty[i]) { memset(&st[i], 0, sizeof st[i]); st[i].frame_offset = ds[i].frame_offset; }
        rc = s2_bank_set_state(nb, st.data());
        if (rc) { s2_bank_destroy(nb); return rc; }
        s2_bank_destroy(s->bank);
        s->bank = nb;
        s->sample_rate = sample_rate;
        for (int i = 0; i < kNumVoices; i++) s->dirty[i] = false;
    }
    if (!s->bank) {
        int rc = s2_bank_create(s->device, sample_rate, s->patch.filter_kind, kNumVoices, s->pending, nullptr, &s->bank);
        if (rc) return rc;
        s->sample_rate = sample_rate;
        for (int i = 0; i < kNumVoices; i++) s->dirty[i] = false;
    }
    return synth_flush(s);
}

int s2_synth_sample(s2_synth* s, float* h_buffer, size_t frames, uint32_t sample_rate) {
    if (!s || (!h_buffer && frames)) return fail(S2_ERR_INVALID, "null argument");
    if (frames == 0) return S2_OK;
    if (sample_rate == 0) return fail(S2_ERR_INVALID, "sample_rate must be > 0");
    int rc = synth_ensure_bank(s, sample_rate);
    if (rc) return rc;
    return s2_bank_render_bus_host(s->bank, frames, nullptr, 0, h_buffer);
}

int s2_synth_set_patch(s2_synth* s, const s2_patch* patch) {
    if (!s || !patch) return fail(S2_ERR_INVALID, "null argument");
    if (patch->filter_kind > S2_FILTER_FIRST_ORDER_HP) return fail(S2_ERR_INVALID, "filter_kind %u", patch->filter_kind);
    s2_voice_desc probe = patch->voice;
    probe.pitch_hz = 440.0f;                    // the template's pitch is replaced per note
    int rc = validate_voice(probe, 0, patch->filter_kind);
    if (rc) return rc;
    if (patch->filter_kind != s->patch.filter_kind) {
        // a voice sounds from its note_on until its amp envelope has ended: release start = max(release, A + D)
        // (old/simdtest.rs:283-285), end = start + R; `has_current` alone never clears (synth.rs:23-30)
        for (int i = 0; i < kNumVoices; i++) {
            const SynthVoice& v = s->voices[i];
            if (!v.has_current) continue;
            bool sounding = !v.has_release;
            if (v.has_release) {
                const s2_voice_desc& d = s->pending[i];
                const double sr = s->sample_rate ? (double)s->sample_rate : 48000.0;
                const double ad = sr * ((double)d.amp_attack_ms + (double)d.amp_decay_ms) / 1000.0;
                const double end = std::max((double)v.release, ad) + sr * (double)d.amp_release_ms / 1000.0 + 1.0;
                sounding = (double)synth_current(s, i) < end;
            }
            if (sounding) return fail(S2_ERR_INVALID, "the filter kind can only change while no voice is sounding");
        }
        s2_bank_destroy(s->bank);               // the next render builds a bank of the new kind
        s->bank = nullptr;
        for (int i = 0; i < kNumVoices; i++) { s2_default_voice(&s->pending[i]); s->dirty[i] = false; s->voices[i] = SynthVoice(); }
    }
    s->patch = *patch;
    s->patch.name[sizeof s->patch.name - 1] = 0;
    return S2_OK;
}

// main.rs:138-147: messages are applied between 16-frame chunks, i.e. before the first chunk that starts at
// or after their arrival
static uint64_t score_quantise(uint64_t frame) { return (frame + 15u) & ~(uint64_t)15u; }

int s2_synth_render_score(s2_synth* s, const s2_note_event* events, size_t n_events, uint32_t sample_rate,
                          float* h_buffer, size_t frames) {
    if (!s || (!h_buffer && frames) || (!events && n_events)) return fail(S2_ERR_INVALID, "null argument");
    if (sample_rate == 0) return fail(S2_ERR_INVALID, "sample_rate must be > 0");
    for (size_t i = 0; i < n_events; i++) {
        if (i && events[i].frame < events[i - 1].frame) return fail(S2_ERR_INVALID, "event %zu is out of time order", i);
        if (events[i].on > 1) return fail(S2_ERR_INVALID, "event %zu: on must be 0 or 1", i);
        if (events[i].frame > 0xFFFFFFFFFFFFFFF0ull) return fail(S2_ERR_INVALID, "event %zu: time out of range", i);
    }
    if (frames == 0) return S2_OK;
    CUDA_TRY(cudaSetDevice(s->device));
    { int rc = grow(s->bank, &s->d_score, 1, s->score_cap, frames); if (rc) return rc; }
    size_t pos = 0, i = 0;
    while (pos < frames) {
        while (i < n_events && score_quantise(events[i].frame) <= pos) {
            const int rc = events[i].on ? s2_synth_note_on(s, events[i].note, events[i].velocity)
                                        : s2_synth_note_off(s, events[i].note);
            if (rc < 0) return rc;
            i++;
        }
        size_t next = frames;
        if (i < n_events && score_quantise(events[i].frame) < frames) next = (size_t)score_quantise(events[i].frame);
        int rc = synth_ensure_bank(s, sample_rate);          // uploads the voices the events touched
        if (rc) return rc;
        rc = bank_render_impl(s->bank, next - pos, nullptr, 0, s->d_score + pos, s2::TRACE_NONE);
        if (rc) return rc;
        pos = next;
    }
    CUDA_TRY(cudaMemcpyAsync(h_buffer, s->d_score, frames * sizeof(float), cudaMemcpyDeviceToHost, s->bank->stream));
    CUDA_TRY(cudaStreamSynchronize(s->bank->stream));
    return S2_OK;
}

int s2_synth_voice_info(s2_synth* s, int slot, uint8_t* note, uint32_t* current_offset_out,
                        uint32_t* release_offset, s2_voice_state* state) {
    if (!s || slot < 0 || slot >= kNumVoices) return fail(S2_ERR_INVALID, "bad slot");
    const SynthVoice& v = s->voices[slot];
    if (note) *note = v.note;
    if (current_offset_out) *current_offset_out = synth_current(s, slot);
    if (release_offset) *release_offset = v.has_release ? v.release : S2_NO_RELEASE;
    if (state) {
        memset(state, 0, sizeof *state);
        if (s->bank && !s->dirty[slot]) {
            std::vector<s2_voice_state> st(kNumVoices);
            int rc = s2_bank_get_state(s->bank, st.data());
            if (rc) return rc;
            *state = st[slot];
        }
    }
    return v.has_current ? 1 : 0;
}

}  // extern "C"
