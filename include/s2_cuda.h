/*
 * s2_cuda.h — C ABI of libs2cuda.so: the B200 (sm_100a) renderer for synth2's hot path
 * (oscillator -> filter -> envelope -> mix, s2_lib/src/try3/{process,synth}.rs).
 *
 * The reference has no FFI of its own (SURVEY.md section 8b): its boundary is the public Rust API of
 * `s2_lib::try3`.  Each entry point below names the reference item it replaces; INTEGRATION.md
 * shows the `extern "C"` block and the safe Rust wrapper (`Synth::new/note_on/note_off/sample`
 * with the reference's signatures) that a maintainer adds to s2_lib to switch the path over.
 *
 * Conventions: plain pointers and sizes only; every call returns S2_OK (0) or a negative
 * S2_ERR_* code and records a message readable through s2_last_error(); no exception crosses
 * the boundary.  A handle is not thread-safe (same contract as `&mut self` in the reference).
 * There is NO CPU fallback: without a CUDA device every compute entry fails with
 * S2_ERR_NO_DEVICE / S2_ERR_CUDA.
 */
#ifndef S2_CUDA_H
#define S2_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define S2_ABI_VERSION 1u

enum {
    S2_OK = 0,
    S2_ERR_INVALID = -1,     /* bad argument (null handle, misaligned buffer, bad enum, ...) */
    S2_ERR_NO_DEVICE = -2,   /* no CUDA device / device index out of range */
    S2_ERR_CUDA = -3,        /* a CUDA runtime call or kernel failed; see s2_last_error() */
    S2_ERR_OVERFLOW = -4,    /* frame offset would pass u32::MAX (reference panics: process.rs:36,71) */
    S2_ERR_NOMEM = -5
};

/* static_config.rs:25-31 `OscillatorKind`, declaration order */
enum { S2_OSC_SQUARE = 0, S2_OSC_SAW = 1, S2_OSC_TRIANGLE = 2, S2_OSC_SINE = 3 };

/* Voice filter.  ONE_POLE is the live reference filter (filters.rs:15-34, driven per sample at
   process.rs:363-371).  BIQUAD_LP is `SecondOrderLowPassFilter` (dsp_filters.rs:82-130), which
   the reference declares but never calls; it is offered for BASELINE config 3.  The rest of that file
   (SURVEY.md 8f row 4, equally uncalled in the reference): BIQUAD_HP = `SecondOrderHighPassFilter`
   (dsp_filters.rs:132-178), BIQUAD_BP = `SecondOrderBandPassFilter` (:180-230; the voice's `damping` field
   carries its quality factor, `lpf_freq_hz` its centre frequency), FIRST_ORDER_LP / _HP =
   `FirstOrderLowPassFilter` / `FirstOrderHighPassFilter` (:12-80; `damping` unused).  In every case the
   cutoff follows the mod envelope exactly as the low-pass's does (process.rs:148-152). */
enum { S2_FILTER_ONE_POLE = 0, S2_FILTER_BIQUAD_LP = 1, S2_FILTER_BIQUAD_HP = 2, S2_FILTER_BIQUAD_BP = 3,
       S2_FILTER_FIRST_ORDER_LP = 4, S2_FILTER_FIRST_ORDER_HP = 5 };

#define S2_NO_RELEASE 0xFFFFFFFFu /* release_frame_offset == None (synth.rs:28; simdtest.rs:283) */

/*
 * One voice = one `sc::Layer` patch (static_config.rs:3-44) + the per-voice fields of
 * `synth::Voice` (synth.rs:23-30).  Times in milliseconds, frequencies in Hz, exactly the
 * reference's units (units.rs:1-17).  80 bytes, no padding.
 */
typedef struct s2_voice_desc {
    uint32_t osc_kind;            /* sc::Oscillator.kind */
    uint32_t noise_seed;          /* st::NoiseState.seed (state.rs:17-21; Synth always uses 0) */
    float pitch_hz;               /* note_to_pitch(note), synth.rs:208-212; see s2_note_to_pitch */
    float osc_gain;               /* sc::Oscillator.gain  (ADDED in the x16 path, process.rs:341-345) */
    float noise_amt;              /* sc::Layer.noise      (ADDED in the x16 path, process.rs:353-356) */
    float lpf_freq_hz;            /* sc::LowPassFilter.freq */
    float damping;                /* BIQUAD_LP only: damping_factor, dsp_filters.rs:94-96 */
    float amp_attack_ms, amp_decay_ms, amp_sustain, amp_release_ms; /* sc::Layer.amp_env */
    float mod_attack_ms, mod_decay_ms, mod_sustain, mod_release_ms; /* sc::Layer.mod_env */
    float mod_env_to_osc_freq;    /* sc::Modulations, Bipolar<10> */
    float mod_env_to_lpf_freq;
    uint32_t frame_offset;        /* Voice.current_frame_offset at the first rendered frame */
    uint32_t release_offset;      /* Voice.release_frame_offset or S2_NO_RELEASE */
    uint32_t active;              /* current_frame_offset.is_some(); 0 = silent, not advanced */
} s2_voice_desc;

/* Carried DSP state of one voice: st::Layer (state.rs:8-21) + Voice.current_frame_offset.
   This is what crosses buffer boundaries; get/set it to checkpoint or migrate a bank. 32 bytes. */
typedef struct s2_voice_state {
    float phase;            /* OscillatorState.phase_accum value (oscillators.rs:402-406) */
    uint32_t has_phase;     /* ... and its Option discriminant (None renders as phase 0.0, process.rs:316) */
    uint32_t frame_offset;  /* advances by `frames` per render, saturating (synth.rs:197) */
    float lpf_last;         /* LowPassFilterState.last (filters.rs:3-7) */
    float x1, x2, y1, y2;   /* SecondOrderLowPassFilterState (dsp_filters.rs:74-80) */
} s2_voice_state;

typedef struct s2_bank s2_bank;   /* V independent voices resident on one GPU */
typedef struct s2_synth s2_synth; /* mirror of synth::Synth (synth.rs:9-12): 8 voices, default patch */

/* ---- library ---- */
uint32_t s2_abi_version(void);
const char* s2_last_error(void);          /* thread-local, never NULL */
int s2_device_count(int* count);

/* synth.rs:208-212 `note_to_pitch` (host libm powf, the same call the reference makes) */
float s2_note_to_pitch(uint8_t note);
/* synth.rs:125-152 `Synth::default_config()` as a voice description (inactive, offset 0) */
void s2_default_voice(s2_voice_desc* out);

/* ---- voice bank: the batched form of process::process_layer_buf_simd (process.rs:14-49) ---- */

/* Uploads `n_voices` descriptions to GPU `device`; `stream` is a cudaStream_t (NULL = default
   stream) on which all work of this bank is enqueued. */
int s2_bank_create(int device, uint32_t sample_rate, uint32_t filter_kind, size_t n_voices,
                   const s2_voice_desc* voices, void* stream, s2_bank** out);
/*
 * Mixed-filter bank: voice i renders through filter filter_kinds[i] (S2_FILTER_*).  Otherwise exactly
 * s2_bank_create.  One bank then holds any patch the library renders (a sweep over filter types, a multitimbral
 * host's parts), and one kernel launch renders every kind.
 *   - Kinds are fixed per voice for the bank's life.  Every other entry (set_voice, set_voices, release_voice,
 *     set_releases, get/set state, trace, pipelining, meters, s2_bank_reduce_bus) works unchanged; a note-on keeps
 *     the voice's kind.  To change kinds, build a new bank (get/set state migrates the voices).
 *   - Validation uses each voice's own kind: damping > 0 is required of second-order voices only.  A bad kind, a NULL
 *     filter_kinds or a bad voice returns S2_ERR_INVALID before anything is allocated.
 *   - Rows, meters and carried state of each voice are bit-identical to those of the same voice in a bank of its kind
 *     made by s2_bank_create, given the same calls in the same order, in every mode.
 *   - Bus: banks of up to 32 voices add in the reference's order, sequentially from 0.0 in voice order, in every
 *     mode; with more than one kind the rows are rendered first (into an internal scratch when d_voice_out is NULL)
 *     and added by one more kernel launch.  Wider banks: as s2_bank_render (deterministic, the same bits in the
 *     default and pipelined modes, in no particular voice order).
 *   - A mixed bank whose voices all share one kind is s2_bank_create with that kind, bit for bit.
 *   - Voices are grouped by kind into whole warps of 32 slots, so a bank of K kinds may hold up to 31 * (K - 1)
 *     padding slots.  The pipelined voice ranges are cut in slots: a narrow bank with several kinds may have more
 *     non-empty ranges, so more launches per render, than a bank of one kind of the same width.
 *   - s2_bank_set_time_split(bank, 1) on a bank of more than one kind returns S2_ERR_INVALID.
 */
int s2_bank_create_mixed(int device, uint32_t sample_rate, size_t n_voices, const s2_voice_desc* voices,
                         const uint32_t* filter_kinds, void* stream, s2_bank** out);
/*
 * Routed bank: voice i renders through filter_kinds[i] and mixes into bus bus_of_voice[i] < n_buses.  Otherwise
 * exactly s2_bank_create_mixed.  A multitimbral host gets one mono signal per part from one bank, one launch per
 * render and one reduction launch per summation form, however many buses there are.
 *   - 1 <= n_buses <= S2_MAX_BUSES.  A NULL bus_of_voice, a bus >= n_buses, a bad kind or a bad voice returns
 *     S2_ERR_INVALID before anything is allocated or any device is touched.  A bus with no voices is allowed: it is
 *     written as +0.0 at every frame.
 *   - A voice's bus and kind are fixed for the bank's life; a note-on keeps both.  Every other entry works unchanged
 *     (set_voice(s), release_voice, set_releases, get/set state, trace, pipelining, time-split, meters,
 *     s2_bank_reduce_bus).  To move a voice to another bus, build a new bank (get/set state migrates the voices).
 *   - Bus g of s2_bank_render_buses is bit-identical to the d_bus_out of a bank made by s2_bank_create_mixed from bus
 *     g's voices alone (same kinds, voices in the same relative order), given the same calls in the same order: at
 *     every bus width, in the default, pipelined and time-split modes, with or without rows and meters.  So a bus of
 *     up to 32 voices adds in the reference's order, sequentially from +0.0 in voice order.  Rows, meters and carried
 *     state of each voice are bit-identical to those of the same voice in that bank.
 *   - s2_bank_render's d_bus_out is the mono sum of all voices, as for a mixed bank: up to 32 voices in voice order;
 *     wider banks a deterministic sum (the same bits in every mode) of per-warp partials by the documented trees, a
 *     warp whose bus has at most 32 voices adding its voices in slot order.
 *   - Layout: each bus's voices are laid out as that standalone bank's, and each bus but the last non-empty one is
 *     padded to whole warps.  Voices are thus grouped into whole warps per (bus, kind): a bank of B buses and K kinds
 *     may hold up to 31 * (B * K - 1) padding slots.  Time-split mode takes routed banks of one kind, as any bank.
 *   - n_buses = 1 makes the bank s2_bank_create_mixed would make.
 */
#define S2_MAX_BUSES 65536u
int s2_bank_create_routed(int device, uint32_t sample_rate, size_t n_voices, const s2_voice_desc* voices,
                          const uint32_t* filter_kinds, const uint32_t* bus_of_voice, uint32_t n_buses,
                          void* stream, s2_bank** out);
void s2_bank_destroy(s2_bank* bank);
size_t s2_bank_voices(const s2_bank* bank);
/* n_voices entries, in voice order.  Works for every bank: a single-kind bank reports its kind for every voice. */
int s2_bank_filter_kinds(const s2_bank* bank, uint32_t* out);
/* *n_buses, and bus_of_voice[n_voices] in voice order (either may be NULL).  Every bank: a bank that is not routed
   has one bus, bus 0. */
int s2_bank_buses(const s2_bank* bank, uint32_t* n_buses, uint32_t* bus_of_voice);

/* Replace one voice (note_on into slot `index`, synth.rs:61-70: fresh state, offset from desc). */
int s2_bank_set_voice(s2_bank* bank, size_t index, const s2_voice_desc* voice);
/* Bulk note_on (synth.rs:61-70 for many voices): entry j replaces voice indices[j] with voices[j], with the same
   effect as s2_bank_set_voice(bank, indices[j], &voices[j]) called for j = 0, 1, ..., n-1.  A repeated index: the
   last entry wins.  Host arrays, copied before the call returns.  Every entry is validated first; on error nothing
   changes.  Asynchronous in every mode: it never waits for the bank's renders.  n = 0 does nothing. */
int s2_bank_set_voices(s2_bank* bank, size_t n, const uint32_t* indices, const s2_voice_desc* voices);
/* note_off for slot `index` (synth.rs:72-80): release_frame_offset = current_frame_offset. */
int s2_bank_release_voice(s2_bank* bank, size_t index);

/* Bulk note_off table: release_frame_offset of every voice (S2_NO_RELEASE = still held), one
   H2D copy of n_voices u32 from `h_release` (pinned memory makes it asynchronous).  This is the
   per-buffer event upload of a streaming caller (main.rs:138-147 applies MIDI, then samples). */
int s2_bank_set_releases(s2_bank* bank, const uint32_t* h_release);

/*
 * Render `frames` frames of every active voice, process_layer_buf_simd semantics per voice
 * (x16 blocks, then `frames % 16` scalar-path tail frames), and advance the carried state.
 *   d_voice_out  device pointer or NULL; row v = d_voice_out + v*row_stride, `frames` floats;
 *                16-byte aligned base and row_stride % 4 == 0.  Inactive voices write zeros.
 *   d_bus_out    device pointer or NULL; `frames` floats, mono (audio_player.rs:23-24):
 *                bus[i] = sum over voices (synth.rs:176-202).  Banks of up to 32 voices add
 *                in exactly the reference's order, in every mode: sequentially from 0.0 in
 *                voice order.  Wider banks add per-warp partials, each a fixed tree over the
 *                warp's 32 slots (slots are voices reordered at creation), then the partials
 *                by a fixed reduction tree; time-split blocks above 32 voices add the rows by
 *                a fixed tree.  Deterministic (the same state and frames give the same bits;
 *                the default and pipelined paths also give the same bits as each other), but
 *                in no particular voice order.
 * Asynchronous on the bank's stream.
 */
int s2_bank_render(s2_bank* bank, size_t frames, float* d_voice_out, size_t row_stride,
                   float* d_bus_out);

/*
 * Per-voice level meters.  Same as s2_bank_render, and for every active voice v also accumulates, in caller voice
 * order:
 *   d_sum_sq[v] += sum over this call's frames of y*y          (binary64 array, 8-byte aligned)
 *   d_peak[v]    = max(d_peak[v], |y|) compared as magnitude bits (binary32 array, 4-byte aligned)
 * d_voice_out and d_bus_out may both be NULL (meters only: no per-voice stores at all).
 *
 * The caller owns both device arrays (n_voices entries each); zeroing them starts a window (a block, a whole render,
 * ...).  Note-ons, releases and state edits never touch them: a meter follows the voice index, not the note.
 *   peak     exact: bits(peak) = max_u32(bits(peak), bits(y) & 0x7fffffff) over every rendered frame, the
 *            `frames % 16` scalar-tail frames included, so a NaN sample ranks above +inf and reads back as NaN (a
 *            second-order filter whose cutoff passes Nyquist blows up; a sweep wants to see it).
 *   sum_sq   within 1e-6 relative of the exact sum of squares while every |y| < 2^64; non-finite once a square
 *            overflows binary32 or a sample is NaN.  Deterministic: squares in binary32, a fixed pairwise tree over
 *            each 64-frame tile counted from the call's first frame, tile totals added in binary64 to a per-call
 *            total that is added to the meter.  Its bits depend only on the voice's parameters and state, `frames`
 *            and the prior meter: the same with or without rows and bus, in the default and the pipelined modes.
 * Inactive voices (and padding) leave their entries bit for bit unchanged.  Asynchronous on the bank's stream;
 * pipelined, each voice range updates its own voices on its own stream, and the meters are complete after
 * s2_bank_sync / s2_bank_join, like the rows.  Time-split mode: a metered block takes the default path (it is not
 * counted by s2_bank_time_split_blocks).  A metered render issues the same kernel launches as the same plain render
 * (in time-split mode: as the plain render on the default path).
 * A NULL bank, a NULL meter or a misaligned meter returns S2_ERR_INVALID with nothing enqueued; every other check
 * is s2_bank_render's.
 */
int s2_bank_render_metered(s2_bank* bank, size_t frames, float* d_voice_out, size_t row_stride,
                           float* d_bus_out, double* d_sum_sq, float* d_peak);

/*
 * Every bus of a bank (s2_bank_create_routed): s2_bank_render, or s2_bank_render_metered when d_sum_sq and d_peak are
 * both set, with bus g written to d_buses + g * bus_stride (`frames` floats each) instead of one d_bus_out.  A bank
 * that is not routed has one bus: its d_bus_out.
 *   d_buses      device pointer, 16-byte aligned, bus_stride % 4 == 0 and bus_stride >= frames (the d_voice_out rules).
 *   d_sum_sq, d_peak   both NULL or both set, as s2_bank_render_metered.
 * Each bus's bits: see s2_bank_create_routed.  A render issues the render launches of s2_bank_render and at most three
 * reduction launches (time-split blocks: two), for any number of buses.
 * Multi-GPU: with bus_stride == frames the buses are one contiguous [n_buses][frames] array, and
 * s2_bank_reduce_bus(bank, comm, root, d_buses, d_out, frames * n_buses, stream) sums them all across the GPUs in one
 * collective call.
 * A NULL bank, a NULL or misaligned d_buses, a bad bus_stride, one meter without the other or a misaligned meter
 * returns S2_ERR_INVALID with nothing enqueued; every other check is s2_bank_render's.
 */
int s2_bank_render_buses(s2_bank* bank, size_t frames, float* d_voice_out, size_t row_stride,
                         float* d_buses, size_t bus_stride, double* d_sum_sq, float* d_peak);

/* Same, then copies the bus to HOST memory and synchronises the stream (Synth::sample shape). */
int s2_bank_render_bus_host(s2_bank* bank, size_t frames, float* d_voice_out, size_t row_stride,
                            float* h_bus_out);

/* Streaming form: enqueues the same work (render, mix, device->host copy of the mix into PINNED host
   memory) and returns without synchronising, so a caller can keep two buffers in flight exactly like
   the reference's player does (audio_player.rs:56-60, sync_channel(2)): enqueue buffer i+1, then wait
   for buffer i (an event on the bank's stream, or s2_bank_sync).  `h_pinned_bus_out` must stay valid
   until then. */
int s2_bank_render_bus_host_async(s2_bank* bank, size_t frames, float* d_voice_out, size_t row_stride,
                                  float* h_pinned_bus_out);

/*
 * Pipelined mode.  n_sub > 1 cuts the bank into n_sub contiguous voice ranges, each rendered on an
 * internal stream, so consecutive s2_bank_render calls overlap across ranges instead of meeting at a
 * device-wide barrier after every block (voices are independent: synth.rs:177-199).  Contract in this mode:
 *   - render calls return at once and are ordered among themselves; their outputs are complete after
 *     s2_bank_sync(), or, on a stream of the caller's, after s2_bank_join(bank, stream);
 *   - the caller must not reuse an output buffer the bank may still be writing (join first);
 *   - s2_bank_set_releases is pipelined too (each range applies the table before its next render), and
 *     so is s2_bank_set_voices (each range that receives entries writes them between its renders);
 *     every other entry (set_voice, release_voice, get/set_state, trace) drains the pipeline first;
 *   - edits take effect in call order, as in the default mode: set_voice, release_voice, a trace or a
 *     pipeline change after s2_bank_set_releases applies the table first, and s2_bank_set_voices writes
 *     its release offsets into a table staged before it, so a later edit of a voice's note-off is never
 *     overwritten by an earlier table;
 *   - s2_bank_trace_phase returns after its render has finished;
 *   - s2_bank_render_bus_host_async makes the bank's own stream (given at creation) wait for the copy.
 * n_sub = 1 (default) keeps everything on the bank's stream.
 */
int s2_bank_set_pipeline(s2_bank* bank, int n_sub);
int s2_bank_join(s2_bank* bank, void* stream);

/*
 * Time-split mode for narrow banks (BASELINE config 2: 1,024 voices, 4,096-frame buffers).
 * With one voice per lane a bank of a thousand voices leaves most of the GPU idle; enable = 1 lets blocks
 * whose voices all hold one period (no pitch modulation) and whose length is a multiple of 1,024 frames
 * render as 32 time segments per voice (with per-frame filter coefficients where a cutoff follows a ramping
 * mod envelope, constant ones otherwise): the
 * oscillator phase is stepped alone and exactly (try3/oscillators.rs:377-381, bit-exact as always), the
 * filter state — one-pole `last` (try3/filters.rs:15-34) or the (y1, y2) of the second-order low-pass
 * (try3/dsp_filters.rs:116-128) — enters each segment through a prefix scan of the segments' affine maps.
 * Output differs from the one-lane-per-voice render only by that scan's reassociation (north star
 * tolerance), so, unlike the default path, a block is not bit-identical to the same frames rendered as two
 * half blocks.  A mix, when requested, is the sum of the rendered rows in voice order (so the rows must be
 * requested too).  Blocks that do not qualify (and every trace request) take the default path;
 * s2_bank_time_split_blocks counts the blocks that did.  Banks of at most 16,384 voices only; exclusive
 * with s2_bank_set_pipeline(n_sub > 1); filter kinds ONE_POLE and BIQUAD_LP.
 */
int s2_bank_set_time_split(s2_bank* bank, int enable);
int s2_bank_time_split_blocks(s2_bank* bank, uint64_t* blocks);

/*
 * Master bus across GPUs (BASELINE config 4; SURVEY.md 8b "s2_bank_reduce_bus(comm, ...)", 8e).  Voices are
 * independent (synth.rs:177-199), so a bank shards as contiguous voice ranges, one bank per GPU, and the only
 * exchange is this: ONE reduce (sum) of the per-GPU buses into the root's master buffer over NCCL / NVLink, once per
 * render (or per >= 1 s chunk), never per block.  The reference has no collective; its mix loop is
 * synth.rs:171-203 and the sum order across GPUs is the collective's (tolerance, not bit-for-bit).
 *   s2_comm_unique_id   ncclGetUniqueId: 128 bytes made on one rank and shipped to the others by the host's own means
 *   s2_comm_create      ncclCommInitRank on `device` (collective: every rank calls it)
 *   s2_comm_adopt       wraps an ncclComm_t the host already owns (not destroyed by s2_comm_destroy)
 *   s2_bank_reduce_bus  joins the bank's internal streams into `stream` (a cudaStream_t, NULL = default), then
 *                       ncclReduce(d_bus_in -> d_bus_out on `root`, f32 sum) on it.  d_bus_out may be NULL off-root
 *                       and may equal d_bus_in.  Asynchronous.
 * NCCL is loaded at run time (dlopen libnccl.so.2); without it these return S2_ERR_NO_DEVICE.
 */
#define S2_COMM_UNIQUE_ID_BYTES 128
typedef struct s2_comm s2_comm;
int s2_comm_version(int* version);
int s2_comm_unique_id(uint8_t* id /* [S2_COMM_UNIQUE_ID_BYTES] */);
int s2_comm_create(const uint8_t* id, int n_ranks, int rank, int device, s2_comm** out);
int s2_comm_adopt(void* nccl_comm, int n_ranks, int rank, int device, s2_comm** out);
void s2_comm_destroy(s2_comm* comm);
int s2_bank_reduce_bus(s2_bank* bank, s2_comm* comm, int root, const float* d_bus_in, float* d_bus_out, size_t frames,
                       void* stream);

/* Checkpoint / restore / test hook.  Host arrays of n_voices entries; synchronises. */
int s2_bank_get_state(s2_bank* bank, s2_voice_state* out);
int s2_bank_set_state(s2_bank* bank, const s2_voice_state* in);
int s2_bank_sync(s2_bank* bank);

/* Debug tap for parity of discrete quantities: renders like s2_bank_render with no output but
   records, per voice and frame, the oscillator phase used for that frame (x16 frames only). */
int s2_bank_trace_phase(s2_bank* bank, size_t frames, float* d_phase_out, size_t row_stride);

/* Number of kernel launches issued through this library by the calling process (bench.py's
   `gpu_launches`). */
uint64_t s2_launch_count(void);

/* ---- Synth mirror (synth.rs:53-203) ---- */
int s2_synth_new(int device, s2_synth** out);                         /* Synth::new()  synth.rs:54-59 */
void s2_synth_free(s2_synth* synth);
int s2_synth_note_on(s2_synth* synth, uint8_t note, float velocity);  /* synth.rs:61-70 */
int s2_synth_note_off(s2_synth* synth, uint8_t note);                 /* synth.rs:72-80; a note no voice holds (or one already released) is ignored */
/* Synth::sample(&mut self, buffer: &mut [f32], sample_rate) synth.rs:154-169: overwrites
   `frames` floats of HOST memory with the mono mix of the 8 voices. */
int s2_synth_sample(s2_synth* synth, float* h_buffer, size_t frames, uint32_t sample_rate);
/* ---- Patch description, note events, offline render (SURVEY.md section 8f rows 1-2) ----
 *
 * The reference's Synth plays one hard-wired patch (`Synth.config` is private and always
 * `default_config()`, synth.rs:10,56,125-152) and is driven 16 frames at a time by `s2_bin`
 * (main.rs:138-147), which applies the MIDI messages that arrived since the previous chunk and then calls
 * `Synth::sample`.  These entries are that loop as one call, plus the patch the `.synth2` file was meant to
 * carry (example.synth2 is an empty `synth mySynth { }`).  Format: synth2_b200/csrc/s2_patch.cpp.
 */
typedef struct s2_patch {
    s2_voice_desc voice;     /* static_config::Layer as a voice template: pitch/offsets/active are ignored */
    uint32_t filter_kind;    /* S2_FILTER_ONE_POLE (the reference's live path) or another S2_FILTER_* */
    char name[60];           /* `synth NAME { ... }` */
} s2_patch;                  /* 144 bytes */

typedef struct s2_note_event {
    uint64_t frame;          /* arrival time in frames from the start of the render */
    uint8_t note;            /* synth::Note */
    uint8_t on;              /* 1 = note_on, 0 = note_off */
    uint8_t reserved[2];
    float velocity;          /* synth::Velocity (Unipolar<1>); stored, never read by the DSP (synth.rs:26) */
} s2_note_event;             /* 16 bytes */

void s2_default_patch(s2_patch* out);     /* Synth::default_config(), one-pole filter, empty name */
/* Parses `.synth2` text.  `events` may be NULL (then the score block is only counted); times given in
   s / ms are converted with `sample_rate`.  Errors carry the line number in s2_last_error(). */
int s2_patch_parse(const char* text, uint32_t sample_rate, s2_patch* out, s2_note_event* events,
                   size_t events_cap, size_t* n_events);
/* Notes started after this call play `patch` (notes already sounding keep theirs).  A change of filter kind
   rebuilds the voice bank and is only allowed while no voice is sounding. */
int s2_synth_set_patch(s2_synth* synth, const s2_patch* patch);
/* Renders `frames` frames of mono mix into HOST memory, applying each event before the first 16-frame chunk
   that starts at or after its arrival time (the s2_bin loop: main.rs:138-147; a 2048-frame player buffer is
   128 such chunks).  Events must be in time order; events at or beyond `frames` are not applied.  The mix is
   rendered into a device buffer, one launch per stretch between events, and copied back once. */
int s2_synth_render_score(s2_synth* synth, const s2_note_event* events, size_t n_events, uint32_t sample_rate,
                          float* h_buffer, size_t frames);

/* ---- Player hand-off (SURVEY.md section 8f row 3): s2_bin/src/audio_player.rs without the cpal device ----
 *
 * Two mono buffers of S2_PLAYER_BUFFER_FRAMES frames (audio_player.rs:21-24) circulate between an internal
 * synth thread (main.rs:120-160: take an empty buffer, apply the note messages that arrived, render, hand
 * it over) and the caller's audio callback.  s2_player_fill is `fill_buffer` (audio_player.rs:136-199) for
 * f32 output: drain the buffer in hand, take at most one new filled buffer without blocking, write every
 * sample to all `channels` interleaved channels, zero-fill the rest (an underrun is counted, never waited
 * for).  It returns the number of frames that came from rendered buffers.  note_on / note_off may be called
 * from any thread; fill from one thread at a time.
 */
#define S2_PLAYER_BUFFER_FRAMES 2048
typedef struct s2_player s2_player;
int s2_player_new(int device, uint32_t sample_rate, s2_player** out);     /* idle until s2_player_start */
void s2_player_free(s2_player* player);
int s2_player_set_patch(s2_player* player, const s2_patch* patch);        /* before s2_player_start */
int s2_player_start(s2_player* player);
int s2_player_note_on(s2_player* player, uint8_t note, float velocity);
int s2_player_note_off(s2_player* player, uint8_t note);
int64_t s2_player_fill(s2_player* player, float* out, size_t frames, uint32_t channels);
int s2_player_stats(s2_player* player, uint64_t* buffers_rendered, uint64_t* underruns, uint64_t* frames_played);
/* blocks until `n_rendered` buffers have been handed over (0) or `timeout_ms` passed (1) */
int s2_player_wait_buffers(s2_player* player, uint64_t n_rendered, uint32_t timeout_ms);

/* test hook: slot contents; returns 1 if the slot has a current_frame_offset, 0 if free */
int s2_synth_voice_info(s2_synth* synth, int slot, uint8_t* note, uint32_t* current_offset,
                        uint32_t* release_offset, s2_voice_state* state);

#ifdef __cplusplus
}
#endif
#endif
