"""Synthetic voice banks of BASELINE.json's shapes (SURVEY.md section 8d "synthetic bank generator").

Counter-based and order-free: every field of voice v is a pure function of (v, field index), so a
rank can generate exactly its own voice range and the oracle and the GPU see identical bytes.

    r(v, k) = splitmix64(0x53594E32_00000000 ^ (v << 8) ^ k),   u(v, k) = (r >> 40) / 2^24 in [0, 1)
"""
import numpy as np

from ._lib import FILTER_BIQUAD_BP, NO_RELEASE, OSC_SAW, OSC_SQUARE, VOICE_DESC
from .bank import note_to_pitch

_M = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64)
    with np.errstate(over="ignore"):
        x = (x + np.uint64(0x9E3779B97F4A7C15)) & _M
        z = x
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M
        return z ^ (z >> np.uint64(31))


def _u(v: np.ndarray, k: int) -> np.ndarray:
    r = splitmix64(np.uint64(0x53594E3200000000) ^ (v.astype(np.uint64) << np.uint64(8)) ^ np.uint64(k))
    return (r >> np.uint64(40)).astype(np.float64) / float(1 << 24)


def pitch_table() -> np.ndarray:
    """128-entry f32 table of `note_to_pitch` (synth.rs:208-212), computed once on the host."""
    return np.array([note_to_pitch(n) for n in range(128)], dtype=np.float32)


# mod-env -> cutoff amounts (octaves at full envelope).  The one-pole filter takes any cutoff
# (k = exp(-2*pi*f/sr) just underflows towards 0), so its banks use the reference default of 10
# (synth.rs:150).  The 2nd-order low-pass (dsp_filters.rs:99-109) is only stable below Nyquist:
# 8000 Hz * 2^1.5 = 22.6 kHz < 24 kHz, so biquad banks sweep 1.5 octaves.
MOD_TO_LPF_ONE_POLE = (0.0, 10.0)
MOD_TO_LPF_BIQUAD = (0.0, 1.5)


def make_bank(n_voices: int, render_frames: int, first_voice: int = 0, kinds=(OSC_SAW, OSC_SQUARE),
              mod_to_lpf_choices=MOD_TO_LPF_ONE_POLE, pitches: np.ndarray = None) -> np.ndarray:
    """Voices [first_voice, first_voice + n_voices) of the synthetic bank.

    note in [24, 108]; cutoff log-uniform [100, 8000] Hz; damping uniform [0.2, 1.414]; A, D, R
    uniform [5, 500] ms; S uniform [0.2, 0.9]; mod env 0/200/0/0 ms; mod->lpf drawn from `mod_to_lpf_choices`; mod->osc 0;
    osc gain 1, noise amount 0, noise seed = voice index; oscillator kind cycles through `kinds`
    by voice index; note-on at frame 0; release at 75 % of `render_frames`, rounded down to a
    multiple of 16.
    """
    if pitches is None:
        pitches = pitch_table()
    v = np.arange(first_voice, first_voice + n_voices, dtype=np.uint64)
    b = np.zeros(n_voices, dtype=VOICE_DESC)
    kinds = np.asarray(kinds, dtype=np.uint32)
    b["osc_kind"] = kinds[(v % np.uint64(len(kinds))).astype(np.int64)]
    b["noise_seed"] = (v & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    note = 24 + np.minimum((_u(v, 0) * 85.0).astype(np.int64), 84)
    b["pitch_hz"] = pitches[note]
    b["osc_gain"] = 1.0
    b["noise_amt"] = 0.0
    b["lpf_freq_hz"] = (100.0 * np.exp(_u(v, 1) * np.log(80.0))).astype(np.float32)
    b["damping"] = (0.2 + _u(v, 2) * (1.414 - 0.2)).astype(np.float32)
    b["amp_attack_ms"] = (5.0 + _u(v, 3) * 495.0).astype(np.float32)
    b["amp_decay_ms"] = (5.0 + _u(v, 4) * 495.0).astype(np.float32)
    b["amp_sustain"] = (0.2 + _u(v, 5) * 0.7).astype(np.float32)
    b["amp_release_ms"] = (5.0 + _u(v, 6) * 495.0).astype(np.float32)
    b["mod_attack_ms"] = 0.0
    b["mod_decay_ms"] = 200.0
    b["mod_sustain"] = 0.0
    b["mod_release_ms"] = 0.0
    b["mod_env_to_osc_freq"] = 0.0
    choices = np.asarray(mod_to_lpf_choices, dtype=np.float32)
    b["mod_env_to_lpf_freq"] = choices[np.minimum((_u(v, 7) * len(choices)).astype(np.int64), len(choices) - 1)]
    b["frame_offset"] = 0
    rel = (int(render_frames) * 3 // 4) & ~15
    b["release_offset"] = rel if rel > 0 else NO_RELEASE
    b["active"] = 1
    return b


# ---- BASELINE config 5: patch-variant sweep (SURVEY.md section 8d) -----------------------------------

SWEEP_AXIS = 32                      # 32 cutoffs x 32 dampings x 32 detunes = 32,768 variants per GPU
SWEEP_VARIANTS = SWEEP_AXIS ** 3


def sweep_axes(sample_rate: int = 48000):
    """The three grid axes, as the f32 values both sides use: cutoff log-spaced 100 Hz..12.8 kHz (7 octaves),
    damping linear 0.2..1.414 (dsp_filters.rs:95: 0.2 is the minimum, sqrt(2) neutral), detune linear
    -50..+50 cents."""
    i = np.arange(SWEEP_AXIS, dtype=np.float64) / (SWEEP_AXIS - 1)
    cutoff = (100.0 * np.exp2(7.0 * i)).astype(np.float32)
    damping = (0.2 + (1.414 - 0.2) * i).astype(np.float32)
    cents = -50.0 + 100.0 * i
    return cutoff, damping, cents


def make_sweep_bank(gpu_index: int, render_frames: int, first_variant: int = 0, n_variants: int = None,
                    sample_rate: int = 48000, kind=OSC_SAW) -> np.ndarray:
    """Variants [first_variant, first_variant + n_variants) of GPU `gpu_index`'s share of the sweep.

    Variant id = (cutoff_index * 32 + damping_index) * 32 + detune_index.  Every variant is the default patch
    (synth.rs:125-152: amp ADSR 100/100/0.5/100 ms, mod ADSR 0/200/0/0 ms, gain 1, noise 0, seed 0) played at
    MIDI note 48 + 4 * gpu_index, detuned: pitch = f32(note_to_pitch(note) * 2^(cents/1200)).  The mod envelope
    opens the cutoff by up to 1.5 octaves but never beyond 0.45 * sample_rate (the 2nd-order low-pass is
    unstable above Nyquist): amount = clamp(log2(0.45 * sr / cutoff), 0, 1.5).  Note-on at frame 0, release
    at 75 % of the render rounded down to a multiple of 16.
    """
    if n_variants is None:
        n_variants = SWEEP_VARIANTS - first_variant
    if not (0 <= first_variant and first_variant + n_variants <= SWEEP_VARIANTS):
        raise ValueError("variant range outside the 32 x 32 x 32 grid")
    cutoff, damping, cents = sweep_axes(sample_rate)
    vid = np.arange(first_variant, first_variant + n_variants, dtype=np.int64)
    ci, di, ti = vid // (SWEEP_AXIS * SWEEP_AXIS), (vid // SWEEP_AXIS) % SWEEP_AXIS, vid % SWEEP_AXIS
    note = 48 + 4 * int(gpu_index)
    if not 0 <= note < 128:
        raise ValueError("gpu_index out of range for a MIDI note")
    base = float(np.float32(note_to_pitch(note)))
    b = default_bank(n_variants)
    b["osc_kind"] = kind
    b["pitch_hz"] = (base * np.exp2(cents[ti] / 1200.0)).astype(np.float32)
    b["lpf_freq_hz"] = cutoff[ci]
    b["damping"] = damping[di]
    room = np.log2(0.45 * float(sample_rate) / cutoff[ci].astype(np.float64))
    b["mod_env_to_lpf_freq"] = np.clip(room, 0.0, 1.5).astype(np.float32)
    rel = (int(render_frames) * 3 // 4) & ~15
    b["release_offset"] = rel if rel > 0 else NO_RELEASE
    b["frame_offset"] = 0
    b["active"] = 1
    return b


SWEEP_FILTER_KINDS = 6                # S2_FILTER_ONE_POLE .. S2_FILTER_FIRST_ORDER_HP


def make_mixed_sweep_bank(gpu_index: int, render_frames: int, first_variant: int = 0, n_variants: int = None,
                          sample_rate: int = 48000, kind=OSC_SAW):
    """Config 5's sweep with the filter kind as a fourth axis: the variants of make_sweep_bank, each (cutoff, damping)
    cell of 32 detunes rendered through filter kind `cell % 6` (the cells cycle through the six kinds, and the 32
    detunes of a cell keep one kind, so they still fill one warp with one cutoff trajectory).  Returns (voices,
    filter_kinds).

    Band-pass voices read `damping` as their quality factor Q, and their coefficients need theta / (2 Q) below pi / 2
    (dsp_filters.rs:197-207, tan); they keep a margin of two, theta / (2 Q) <= pi / 4, i.e. a cutoff of at most
    Q * sample_rate / 4: their cutoff is clamped to that limit (and to 0.45 * sample_rate), and their mod amount to
    the room left below it.  The other kinds keep make_sweep_bank's values.
    """
    b = make_sweep_bank(gpu_index, render_frames, first_variant, n_variants, sample_rate, kind)
    vid = np.arange(first_variant, first_variant + b.shape[0], dtype=np.int64)
    kinds = ((vid // SWEEP_AXIS) % SWEEP_FILTER_KINDS).astype(np.uint32)
    bp = kinds == FILTER_BIQUAD_BP
    limit = np.minimum(0.45 * float(sample_rate), b["damping"][bp].astype(np.float64) * float(sample_rate) / 4.0)
    cutoff = np.minimum(b["lpf_freq_hz"][bp].astype(np.float64), limit).astype(np.float32)
    b["lpf_freq_hz"][bp] = cutoff
    b["mod_env_to_lpf_freq"][bp] = np.clip(np.log2(limit / cutoff.astype(np.float64)), 0.0, 1.5).astype(np.float32)
    return b, kinds


def default_bank(n: int) -> np.ndarray:
    """n copies of `Synth::default_config()` (synth.rs:125-152), inactive, as written by the library."""
    from .bank import default_voice
    return default_voice(n)
