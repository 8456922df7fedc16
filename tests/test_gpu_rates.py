"""The render paths away from 48 kHz and at the edges of their parameters.

The sample rate feeds every constant the kernels derive — the oscillator's period and phase step, the envelopes'
stage boundaries (ms * sr / 1000), the angle of a moving cutoff (2 pi f / sr, s2c::theta_of: the IEEE quotient at
the usual rates, within an ulp at any other) and the limits of its 32-frame windows — so the bank paths are checked
here at rates from 8 kHz to 192 kHz, including two (12,345 Hz and 47,999 Hz) that are on no list.  Beyond that:

  * pitches at and above the sample rate, which the fast paths must leave to the general one (they need a phase
    step below 1), and the band [sr / 2, sr) that the fast paths do take;
  * warps whose voices share one cutoff trajectory (one set of coefficients per chunk, computed once per warp), for
    every filter;
  * a one-pole cutoff modulated past the binary32 range (theta = +inf), whose k = e^-theta must be 0 as in the
    reference, not NaN.
"""
import numpy as np
import pytest

import oracle
import synth2_b200 as s2
from synth2_b200 import bankgen
from synth2_b200 import patch as s2patch
from test_gpu_parity import TOL_ABS, assert_parity

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ALL_FILTERS = (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP, s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP,
               s2.FILTER_FIRST_ORDER_LP, s2.FILTER_FIRST_ORDER_HP)
F32 = np.float32


# ------------------------------------------------------------------------------ helpers

def rate_bank(filter_kind, n, sr, frames, seed=0, low_hz=100.0):
    """A bank for any rate and filter.  Cutoffs are drawn so that the sweep of the mod envelope stays inside
    [low_hz * sr / 48000, 0.45 * sr]: the same range of angles the 48 kHz banks cover, so the second-order filters
    stay stable and as well conditioned as there.  Modulation amounts of both signs, and mod-envelope ramps in attack,
    decay and release, so the cutoff moves in all three; amp and mod envelope times scale with the render's
    duration, so stage boundaries land inside the render (and inside chunks) at every rate.  All four oscillators,
    noise on some voices, other gains, inactive voices, start offsets on and off multiples of 32, releases mid-block
    and some voices held."""
    total = int(sum(frames))
    rng = np.random.default_rng(seed * 1000003 + sr + 17 * filter_kind)
    v = bankgen.make_bank(n, total, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE),
                          mod_to_lpf_choices=(0.0,))
    amounts = (0.0, 1.5, -1.0, 0.75, -1.5) + ((10.0,) if filter_kind == s2.FILTER_ONE_POLE else ())
    amt = np.asarray(amounts, np.float64)[rng.integers(0, len(amounts), n)]
    lo = low_hz * sr / 48000.0 * np.exp2(np.maximum(-amt, 0.0))
    hi = 0.45 * sr / np.exp2(np.clip(amt, 0.0, 1.5))
    v["mod_env_to_lpf_freq"] = amt.astype(F32)
    v["lpf_freq_hz"] = (lo * np.exp(rng.uniform(0.0, 1.0, n) * np.log(hi / lo))).astype(F32)
    if filter_kind == s2.FILTER_BIQUAD_BP:
        v["damping"] += 2.0        # the field is the quality factor here; theta / (2 Q) must stay below pi / 4
    dur = 1000.0 * total / sr      # ms
    u = lambda lo_, hi_: rng.uniform(lo_, hi_, n).astype(F32)
    v["amp_attack_ms"] = dur * u(0.005, 0.2)
    v["amp_decay_ms"] = dur * u(0.005, 0.2)
    v["amp_sustain"] = u(0.3, 0.9)
    v["amp_release_ms"] = dur * u(0.03, 0.2)
    v["mod_attack_ms"] = dur * u(0.0, 0.08)
    v["mod_decay_ms"] = dur * u(0.03, 0.25)
    v["mod_sustain"] = u(0.2, 0.8)
    v["mod_release_ms"] = dur * u(0.02, 0.15)
    v["noise_amt"][::3] = 0.25
    v["osc_gain"][::5] = 0.5
    v["active"][7::31] = 0
    v["frame_offset"][n // 2:] = np.array([16, 32, 37, 5, 64, 96, 100], np.uint32)[np.arange(n - n // 2) % 7]
    rel = v["frame_offset"].astype(np.int64) + (total * rng.uniform(0.45, 0.8, n)).astype(np.int64)
    v["release_offset"] = rel.astype(np.uint32)
    v["release_offset"][4::9] = s2.NO_RELEASE
    return v


def gpu_render(voices, sr, filter_kind, blocks, pipeline=1, time_split=False):
    """Consecutive blocks on the GPU: (rows [V, sum blocks], final state, blocks the time-split kernels rendered)."""
    V = voices.shape[0]
    outs = []
    with s2.VoiceBank(voices, sr, filter_kind) as bank:
        if pipeline > 1:
            bank.set_pipeline(pipeline)
        if time_split:
            bank.set_time_split(True)
        for fr in blocks:
            stride = (fr + 3) & ~3
            vo = torch.full((V, stride), float("nan"), device="cuda", dtype=torch.float32)
            bank.render(fr, vo, stride, None)
            bank.sync()
            outs.append(vo[:, :fr].cpu().numpy())
        st = bank.get_state()
        n_ts = bank.time_split_blocks
    return np.concatenate(outs, axis=1), st, n_ts


def gpu_render_paths(voices, sr, filter_kind, blocks, paths, monkeypatch):
    """The same render with S2_FORCE_PATH = each of `paths` (0 default, 1 one frame at a time in moving-cutoff
    chunks, 2 the general per-frame path, 3 packed chunks without lane pairs)."""
    res = {}
    for p in paths:
        monkeypatch.setenv("S2_FORCE_PATH", str(p))
        res[p] = gpu_render(voices, sr, filter_kind, blocks)
    monkeypatch.delenv("S2_FORCE_PATH")
    return res


def oracle_render(voices, sr, filter_kind, blocks):
    st = oracle.bank_init_states(voices)
    outs = []
    for fr in blocks:
        o, _ = oracle.bank_render(voices, st, sr, filter_kind, fr, want_bus=False, nthreads=8)
        outs.append(o)
    return np.concatenate(outs, axis=1), st


def assert_same_bits(a, b, what):
    """Rows and state of two GPU renders are identical."""
    bad = np.argwhere(a[0].view(np.uint32) != b[0].view(np.uint32))
    assert bad.size == 0, f"{what}: first differing (voice, frame): {bad[:5].tolist()}"
    assert a[1].tobytes() == b[1].tobytes(), f"{what}: state"


def assert_state(st, rst, filter_kind, exact_phase=True):
    assert np.array_equal(st["frame_offset"], rst["frame_offset"])
    assert np.array_equal(st["has_phase"], rst["has_phase"])
    if exact_phase:
        assert st["phase"].tobytes() == rst["phase"].tobytes()
    keys = {s2.FILTER_ONE_POLE: ("lpf_last",), s2.FILTER_FIRST_ORDER_LP: ("x1", "y1"),
            s2.FILTER_FIRST_ORDER_HP: ("x1", "y1")}.get(filter_kind, ("x1", "x2", "y1", "y2"))
    for k in keys:
        np.testing.assert_allclose(st[k], rst[k], atol=TOL_ABS * 4, rtol=0, err_msg=k)


def pitches_of(notes):
    return np.array([s2.note_to_pitch(int(n)) for n in notes], F32)


# ------------------------------------------------------------------------------ 1. rate x filter matrix

RATES = (8000, 11025, 12345, 22050, 44100, 47999, 96000, 192000)
BLOCKS = [4096, 4096, 2048, 1000, 3096]


@pytest.mark.parametrize("sr", RATES)
@pytest.mark.parametrize("filter_kind", ALL_FILTERS)
def test_rate_matrix(filter_kind, sr, monkeypatch):
    """Every filter at every rate: against the oracle within the north-star bar, phase and offsets bit-exact, the
    carried filter state; the four kernel paths and three pipelined voice ranges give identical bits."""
    V = 197                                        # a ragged last warp
    v = rate_bank(filter_kind, V, sr, BLOCKS)
    ref, rst = oracle_render(v, sr, filter_kind, BLOCKS)
    assert np.all(np.isfinite(ref))
    outs = gpu_render_paths(v, sr, filter_kind, BLOCKS, (0, 1, 2, 3), monkeypatch)
    got, st, _ = outs[0]
    assert_parity(ref, got, f"filter {filter_kind} at {sr} Hz")
    assert_state(st, rst, filter_kind)
    assert np.all(got[v["active"] == 0] == 0.0)
    for p in (1, 2, 3):
        assert_same_bits(outs[0], outs[p], f"S2_FORCE_PATH={p} at {sr} Hz")
    pipe = gpu_render(v, sr, filter_kind, BLOCKS, pipeline=3)
    assert_same_bits(outs[0], pipe, f"pipeline 3 at {sr} Hz")


@pytest.mark.parametrize("sr", RATES)
@pytest.mark.parametrize("filter_kind", (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP))
def test_rate_matrix_time_split(filter_kind, sr):
    """The time-split kernels at every rate: the blocks of whole 1,024-frame multiples go through them (moving
    cutoffs included), the others fall back.  Against the oracle and the default path; phase bit-exact.

    The second-order low-pass starts each time segment from the state of a binary64 scan, where the reference's
    binary32 recurrence carries its own rounding bias; at the lowest angles that bias alone comes near the bar
    (a resting 204 Hz cutoff at 96 kHz, damping 0.7, put the time-split render 7e-4 off a full scale of 4 while the
    default path matched the oracle bit for bit).  So its cutoffs start at the angle of 300 Hz at 48 kHz here; the
    default-path matrix above covers the lowest angles."""
    V = 197
    low_hz = 300.0 if filter_kind == s2.FILTER_BIQUAD_LP else 100.0
    v = rate_bank(filter_kind, V, sr, BLOCKS, seed=1, low_hz=low_hz)
    ref, rst = oracle_render(v, sr, filter_kind, BLOCKS)
    got, st, n_ts = gpu_render(v, sr, filter_kind, BLOCKS, time_split=True)
    assert n_ts == 3                               # 1000 and 3096 are not multiples of 1,024
    assert_parity(ref, got, f"time-split filter {filter_kind} at {sr} Hz vs oracle")
    assert_state(st, rst, filter_kind)
    plain, st0, n0 = gpu_render(v, sr, filter_kind, BLOCKS)
    assert n0 == 0
    assert st["phase"].tobytes() == st0["phase"].tobytes()
    assert np.array_equal(st["frame_offset"], st0["frame_offset"])
    assert_parity(plain, got, f"time-split filter {filter_kind} at {sr} Hz vs default path")


# ------------------------------------------------------------------------------ 2. extreme pitches

@pytest.mark.parametrize("sr", [8000, 11025])
def test_phase_trace_of_high_notes_at_low_rates(sr):
    """MIDI 100-127 at 8 and 11.025 kHz: above Nyquist, at and above the rate.  The phase before every frame is the
    oracle's, bit for bit."""
    frames = 8192
    notes = list(range(100, 128))
    v = s2.default_voice(len(notes))
    v["active"] = 1
    v["pitch_hz"] = pitches_of(notes)
    v["osc_kind"] = [i % 4 for i in range(len(notes))]
    ph = torch.zeros((len(notes), frames), device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, sr, s2.FILTER_ONE_POLE) as bank:
        bank.trace_phase(frames, ph)
        bank.sync()
    got = ph.cpu().numpy()
    for i, n in enumerate(notes):
        cfg = oracle.default_config()
        cfg["osc_kind"] = v["osc_kind"][i]
        _, rph, _, _ = oracle.trace_voice(cfg, float(v["pitch_hz"][i]), sr, 0, oracle.NO_RELEASE, frames)
        assert got[i].tobytes() == rph.tobytes(), f"note {n} at {sr} Hz"


def edge_pitches(sr):
    """Around Nyquist, around the rate, at it, and above it."""
    sr = float(sr)
    return np.array([sr / 2 * (1 - 2.0 ** -23), sr / 2, sr / 2 * (1 + 2.0 ** -23), sr * (1 - 2.0 ** -24), sr,
                     sr * (1 + 2.0 ** -23), 1.5 * sr, 3.7 * sr], F32)


def test_edge_pitches_bit_exact_in_a_warp_of_ordinary_voices(monkeypatch):
    """At 48 kHz, pitches just below, at and just above Nyquist, just below, at and above the rate, 1.5 and 3.7 times
    it, for every oscillator, in warps with ordinary voices.  With the filter and envelopes transparent
    (k = exp(-huge) = 0, A = D = 0, S = 1) the output is (osc + gain) + (noise + amt): every bit must match the
    oracle, on the default and the general path, through the scalar tail."""
    sr = 48000
    edge = edge_pitches(sr)
    ordinary = pitches_of([45, 60, 69, 81, 93, 100, 57, 64])
    # per oscillator: the 8 edge pitches and 2 ordinary ones; 40 voices, so warp 0 mixes both and warp 1 is ragged
    pitch = np.concatenate([np.concatenate([edge, ordinary[2 * k:2 * k + 2]]) for k in range(4)])
    n = pitch.size
    v = bankgen.make_bank(n, 1 << 16)
    v["osc_kind"] = np.repeat(np.arange(4), n // 4).astype(np.uint32)
    v["pitch_hz"] = pitch
    v["lpf_freq_hz"] = 1.0e9
    v["mod_env_to_lpf_freq"] = 0.0
    v["amp_attack_ms"] = 0.0; v["amp_decay_ms"] = 0.0; v["amp_sustain"] = 1.0
    v["release_offset"] = s2.NO_RELEASE
    v["noise_amt"][::2] = 0.25
    blocks = [4096, 4096, 1000]
    ref, rst = oracle_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    outs = gpu_render_paths(v, sr, s2.FILTER_ONE_POLE, blocks, (0, 2), monkeypatch)
    for p, (got, st, _) in outs.items():
        bad = np.argwhere(got.view(np.uint32) != ref.view(np.uint32))
        assert bad.size == 0, f"path {p}: first differing (voice, frame): {bad[:5].tolist()}"
        assert st["phase"].tobytes() == rst["phase"].tobytes()


@pytest.mark.parametrize("sr", [8000, 48000])
def test_edge_pitches_with_the_default_patch(sr):
    """The default patch (one-pole, the 10-octave cutoff sweep) at edge pitches — at 8 kHz MIDI 108-127, at 48 kHz
    the explicit ones — among ordinary voices: against the oracle, phase bit-exact."""
    if sr == 8000:
        pitch = pitches_of(list(range(108, 128)) + [40, 52, 64, 76, 88])
    else:
        pitch = np.concatenate([edge_pitches(sr), pitches_of([40, 52, 64, 76, 88, 100, 33])])
    n = pitch.size
    v = s2.default_voice(n)
    v["active"] = 1
    v["pitch_hz"] = pitch
    v["osc_kind"] = np.arange(n) % 4
    v["release_offset"] = 6000 + 7 * np.arange(n)
    blocks = [4096, 4096, 2048, 1000]
    ref, rst = oracle_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    got, st, _ = gpu_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    assert_parity(ref, got, f"edge pitches, default patch, {sr} Hz")
    assert_state(st, rst, s2.FILTER_ONE_POLE)


def test_time_split_refuses_a_pitch_at_the_rate():
    """At 8 kHz a voice in [sr / 2, sr) may go through the time-split kernels (phase step in [0.5, 1)); a voice at
    MIDI 124 (10.5 kHz) must not: the host classifier refuses every block, which then renders exactly as the
    default path does."""
    sr = 8000
    blocks = [2048, 2048, 1024]
    v = rate_bank(s2.FILTER_ONE_POLE, 64, sr, blocks, seed=2)
    v["pitch_hz"][10] = s2.note_to_pitch(110)      # 4.7 kHz: above Nyquist, below the rate
    assert v["active"][10] and v["active"][20]
    ref, rst = oracle_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    got, st, n_ts = gpu_render(v, sr, s2.FILTER_ONE_POLE, blocks, time_split=True)
    assert n_ts == 3
    assert_parity(ref, got, "time-split with a pitch above Nyquist")
    assert_state(st, rst, s2.FILTER_ONE_POLE)

    v["pitch_hz"][20] = s2.note_to_pitch(124)      # 10.5 kHz: above the rate
    ref, rst = oracle_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    got, st, n_ts = gpu_render(v, sr, s2.FILTER_ONE_POLE, blocks, time_split=True)
    assert n_ts == 0
    plain = gpu_render(v, sr, s2.FILTER_ONE_POLE, blocks)
    assert_same_bits(plain, (got, st), "refused time-split vs default path")
    assert_parity(ref, got, "time-split refused, pitch above the rate")
    assert_state(st, rst, s2.FILTER_ONE_POLE)


def test_synth_plays_the_top_notes_at_8k():
    """Synth at 8 kHz: notes 118-127 (10 notes into 8 slots: the oldest are stolen), then two note-offs, against
    OracleSynth."""
    sr = 8000
    osyn, syn = oracle.OracleSynth(), s2.Synth()
    a, b = np.zeros(800, np.float32), np.zeros(800, np.float32)
    for note in range(118, 128):
        osyn.note_on(note); syn.note_on(note)
        osyn.sample(a, sr); syn.sample(b, sr)
        assert_parity(a, b, f"after note_on {note}")
    for note in (120, 125):
        osyn.note_off(note); syn.note_off(note)
    a, b = np.zeros(4000, np.float32), np.zeros(4000, np.float32)
    osyn.sample(a, sr); syn.sample(b, sr)
    assert_parity(a, b, "after the note_offs")
    for slot in range(8):
        assert syn.voice_info(slot)[:4] == osyn.voice_info(slot)[:4]
    syn.close()


# ------------------------------------------------------------------------------ 3. warps sharing one cutoff trajectory

SHARED_BLOCKS = [4096, 4096, 2048, 1000, 1032]


def shared_bank(filter_kind, sr):
    """32 voices (a bank this small keeps identity slots: one warp) with one cutoff trajectory — cutoff, damping,
    modulation amount, mod envelope, start offset and release — and different pitches, oscillators, noise and amp
    envelopes.  The start offset is not a multiple of 32; the amp envelopes' stage boundaries fall inside moving
    chunks; the mod envelope ramps in attack, decay and release.  Two lanes are inactive, parked at other offsets
    with another cutoff."""
    n, total = 32, sum(SHARED_BLOCKS)
    rng = np.random.default_rng(sr + filter_kind)
    v = bankgen.make_bank(n, total, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE),
                          mod_to_lpf_choices=(0.0,))
    v["pitch_hz"] = pitches_of(rng.integers(36, 100, n))
    v["lpf_freq_hz"] = F32(0.04 * sr)
    v["mod_env_to_lpf_freq"] = {22050: 1.5, 48000: -1.25, 96000: 1.0}[sr]
    v["damping"] = 0.7 + (2.0 if filter_kind == s2.FILTER_BIQUAD_BP else 0.0)
    v["mod_attack_ms"] = 4.0; v["mod_decay_ms"] = 40.0; v["mod_sustain"] = 0.4; v["mod_release_ms"] = 25.0
    v["frame_offset"] = 37
    v["release_offset"] = 37 + int(0.6 * total) + 5
    v["amp_attack_ms"] = rng.uniform(1.0, 12.0, n).astype(F32)
    v["amp_decay_ms"] = rng.uniform(5.0, 40.0, n).astype(F32)
    v["amp_sustain"] = rng.uniform(0.3, 0.9, n).astype(F32)
    v["amp_release_ms"] = rng.uniform(10.0, 40.0, n).astype(F32)
    v["noise_amt"][3::8] = 0.25
    v["active"][[9, 22]] = 0
    v["frame_offset"][[9, 22]] = [777, 5]
    v["lpf_freq_hz"][[9, 22]] = 1234.0
    return v


@pytest.mark.parametrize("sr", [22050, 48000, 96000])
@pytest.mark.parametrize("filter_kind", ALL_FILTERS)
def test_shared_trajectory_warp(filter_kind, sr, monkeypatch):
    """A warp whose voices share one cutoff trajectory computes each moving chunk's coefficients once: the packed
    and the one-frame-at-a-time forms of that (paths 0 and 1) give the general path's bits (2), and the oracle's
    output within the bar.  With one voice's cutoff changed the warp no longer shares, and every other row keeps
    its bits."""
    v = shared_bank(filter_kind, sr)
    ref, rst = oracle_render(v, sr, filter_kind, SHARED_BLOCKS)
    assert np.all(np.isfinite(ref))
    outs = gpu_render_paths(v, sr, filter_kind, SHARED_BLOCKS, (0, 1, 2), monkeypatch)
    for p in (0, 1):
        assert_same_bits(outs[2], outs[p], f"shared warp, S2_FORCE_PATH={p}, filter {filter_kind} at {sr} Hz")
    got, st, _ = outs[0]
    assert_parity(ref, got, f"shared warp, filter {filter_kind} at {sr} Hz")
    assert_state(st, rst, filter_kind)
    assert np.all(got[v["active"] == 0] == 0.0)

    w = v.copy()
    w["lpf_freq_hz"][13] *= F32(1.1)
    got2, _, _ = gpu_render(w, sr, filter_kind, SHARED_BLOCKS)
    keep = np.arange(32) != 13
    assert got2[keep].tobytes() == got[keep].tobytes()
    ref13, _ = oracle_render(w[13:14], sr, filter_kind, SHARED_BLOCKS)
    assert_parity(ref13, got2[13:14], "the voice that broke the warp")


_FILTER_NAMES = {0: "one_pole", 1: "biquad", 2: "biquad_hp", 3: "biquad_bp", 4: "first_order", 5: "first_order_hp"}


@pytest.mark.parametrize("sr", [44100, 96000])
@pytest.mark.parametrize("filter_kind", ALL_FILTERS)
def test_synth_chord_shares_a_trajectory(filter_kind, sr):
    """A Synth chord started in one call: 8 voices of one patch at offset 0, so one warp with one moving cutoff.
    Expected: each note rendered by the oracle from its note-on, mixed in slot order (what OracleSynth does; for
    the default patch's filter, OracleSynth itself)."""
    damping = 2.6 if filter_kind == s2.FILTER_BIQUAD_BP else 0.8
    text = (f"synth chord {{ osc {{ kind saw }} lpf {{ freq 1500; kind {_FILTER_NAMES[filter_kind]}; "
            f"damping {damping} }} amp_env {{ attack 5; decay 40; sustain 0.6; release 30 }} "
            f"mod_env {{ attack 3; decay 50; sustain 0.3; release 20 }} modulations {{ mod_env_to_lpf_freq 1.5 }} }}")
    p = s2patch.parse(text, sr)
    assert p.filter_kind == filter_kind
    notes = [48, 52, 55, 59, 62, 65, 69, 72]
    n1, n2 = (int(0.1 * sr) // 16) * 16, (int(0.08 * sr) // 16) * 16
    syn = s2.Synth()
    syn.set_patch(p)
    for note in notes:
        syn.note_on(note)
    got = np.zeros(n1 + n2, np.float32)
    syn.sample(got[:n1], sr)
    for note in notes:
        syn.note_off(note)
    part = np.zeros(n2, np.float32)
    syn.sample(part, sr)
    got[n1:] = part
    syn.close()
    mix = np.zeros(n1 + n2, np.float32)
    for note in notes:
        vd = np.zeros(1, dtype=s2.VOICE_DESC)
        vd[0] = p.voice
        vd["pitch_hz"] = s2.note_to_pitch(note)
        vd["active"] = 1
        vd["frame_offset"] = 0
        vd["release_offset"] = n1
        o, _ = oracle.bank_render(vd, oracle.bank_init_states(vd), sr, filter_kind, n1 + n2, want_bus=False)
        mix = mix + o[0]
    assert_parity(mix, got, f"chord, filter {filter_kind} at {sr} Hz")
    assert np.max(np.abs(mix)) > 0.1
    if filter_kind == s2.FILTER_ONE_POLE:
        # the default patch (one-pole, 10-octave sweep) needs no mirror: OracleSynth plays it
        osyn, syn = oracle.OracleSynth(), s2.Synth()
        for note in notes:
            osyn.note_on(note); syn.note_on(note)
        a, b = np.zeros(n1, np.float32), np.zeros(n1, np.float32)
        osyn.sample(a, sr); syn.sample(b, sr)
        assert_parity(a, b, f"default-patch chord at {sr} Hz")
        syn.close()


# ------------------------------------------------------------------------------ 4. cutoffs that overflow binary32

OVERFLOW = [(127.5, None), (128.0, None), (130.0, None), (-130.0, None), (200.0, None), (10.0, 3.0e38),
            (10.0, None)]                          # (mod_env_to_lpf_freq, cutoff or the default's)


def overflow_bank(n, shared=False):
    """One-pole voices of the default patch whose moving cutoff overflows binary32 somewhere in the mod decay:
    2^(m amount) for m amount >= 128, or 2 pi f for f = 3e38 Hz; amount 127.5 stays just inside, -130 underflows,
    and one voice in seven is the default patch.  shared: every voice has amount 130 (one trajectory per warp)."""
    v = s2.default_voice(n)
    v["active"] = 1
    v["pitch_hz"] = pitches_of(40 + (7 * np.arange(n)) % 50)
    v["osc_kind"] = np.arange(n) % 4
    v["release_offset"] = 6000 if shared else 6000 + 3 * np.arange(n)
    if shared:
        v["mod_env_to_lpf_freq"] = 130.0
        return v
    for i in range(n):
        amt, cutoff = OVERFLOW[i % len(OVERFLOW)]
        v["mod_env_to_lpf_freq"][i] = amt
        if cutoff is not None:
            v["lpf_freq_hz"][i] = cutoff
    return v


OVF_BLOCKS = [4096, 4096, 2048, 2048]


def test_overflowing_one_pole_cutoff_is_finite(monkeypatch):
    """k = e^-theta of a one-pole cutoff modulated past binary32 is 0, as the reference's exp(-inf): finite output
    within the bar of the oracle on every path — packed and one-frame moving-cutoff chunks, the general path,
    pipelined voice ranges, the time-split kernels — and in a warp that shares the trajectory.  (The second-order
    and first-order filters are left out: sin and cos of an infinite angle are NaN in the reference as well.)"""
    sr, fk = 48000, s2.FILTER_ONE_POLE
    v = overflow_bank(70)
    ref, rst = oracle_render(v, sr, fk, OVF_BLOCKS)
    assert np.all(np.isfinite(ref))
    outs = gpu_render_paths(v, sr, fk, OVF_BLOCKS, (0, 1, 2), monkeypatch)
    for p, res in outs.items():
        assert_parity(ref, res[0], f"overflowing cutoffs, S2_FORCE_PATH={p}")
        assert_state(res[1], rst, fk)
    for p in (1, 2):
        assert_same_bits(outs[0], outs[p], f"overflowing cutoffs, S2_FORCE_PATH={p}")
    pipe = gpu_render(v, sr, fk, OVF_BLOCKS, pipeline=2)
    assert_same_bits(outs[0], pipe, "overflowing cutoffs, pipeline 2")
    ts, st, n_ts = gpu_render(v, sr, fk, OVF_BLOCKS, time_split=True)
    assert n_ts == len(OVF_BLOCKS)
    assert_parity(ref, ts, "overflowing cutoffs, time-split")
    assert_state(st, rst, fk)

    w = overflow_bank(32, shared=True)
    wref, _ = oracle_render(w, sr, fk, OVF_BLOCKS)
    assert np.all(np.isfinite(wref))
    wouts = gpu_render_paths(w, sr, fk, OVF_BLOCKS, (0, 1, 2), monkeypatch)
    for p, res in wouts.items():
        assert_parity(wref, res[0], f"overflowing shared trajectory, S2_FORCE_PATH={p}")
