"""Pins the CPU oracle against every known-answer the reference holds for this path
(SURVEY.md section 8c): the 4 `#[test]` functions of s2_lib and the notebook prototype values,
plus derived known-answers computed from the reference definitions (labelled *derived*)."""
import pathlib

import numpy as np
import pytest

import oracle

L = oracle.lib()
NONE = oracle.NO_RELEASE


def f32(x):
    return np.float32(x)


# ---- hashnoise.rs:70-98 -------------------------------------------------------------------

def test_hash_word_scalar_equals_x16():
    """hashnoise.rs:70-83 `test_hash_word`."""
    start = np.full(16, 0xFF00FF00, dtype=np.uint32)
    word = np.full(16, 0x11111111, dtype=np.uint32)
    out = np.zeros(16, dtype=np.uint32)
    L.s2o_hash_word_x16(start.ctypes.data, word.ctypes.data, out.ctypes.data)
    h = L.s2o_hash_word(0xFF00FF00, 0x11111111)
    assert h == out[0]
    assert h == 0xB1BDD11E  # derived


def test_hash_word_dist():
    """hashnoise.rs:85-98 `test_hash_word_dist`: sum of popcounts over 200,004 hashes == count * 16."""
    count = 200004
    ones = sum(bin(L.s2o_hash_word(0, i)).count("1") for i in range(count))
    assert ones == count * 16 == 3200064


def test_hash_matches_numpy_restatement():
    i = np.arange(200004, dtype=np.uint64)
    h = (i * np.uint64(0x9E3779B9)) & np.uint64(0xFFFFFFFF)   # rotl(0,5) ^ i == i
    probe = [0, 1, 2, 77, 65535, 65536, 200003]
    for p in probe:
        assert L.s2o_hash_word(0, p) == int(h[p])


# ---- lookup.rs:250-310 --------------------------------------------------------------------

@pytest.mark.parametrize("x16", [1, 0])
def test_table_lookup(x16):
    """lookup.rs:250-279 `test_table_lookup` (x16) and :281-310 `test_table_lookup_x16` (scalar)."""
    t4 = np.array([0, 1, 2, 3], dtype=np.float32)
    t5 = np.array([0, 1, 2, 3, 4], dtype=np.float32)
    ex = lambda v: L.s2o_table_lookup_exclusive(t4.ctypes.data, 4, v, 4.0, x16)
    inc = lambda v: L.s2o_table_lookup_inclusive(t5.ctypes.data, 5, v, 4.0, x16)
    assert ex(0.0) == 0.0
    assert ex(0.5) == 0.5
    assert ex(3.5) == 1.5      # wraps to index 0
    assert inc(0.0) == 0.0
    assert inc(0.5) == 0.5
    assert inc(3.0) == 3.0
    assert inc(4.0) == 4.0


# ---- Untitled.ipynb cells 2 and 4 (f64 prototype; weak known answers) --------------------------

@pytest.mark.parametrize("fn", ["s2o_adsr_x16_lane", "s2o_adsr_scalar"])
def test_notebook_adsr(fn):
    adsr = getattr(L, fn)
    assert adsr(1.0, 100.0, 0.5, 1.0, 10, NONE) == pytest.approx(0.955, abs=1e-6)
    got = [adsr(0.0, 10.0, 0.0, 10.0, n, 30) for n in range(40)]
    want = [1.0 - 0.1 * n for n in range(10)] + [0.0] * 30
    assert got == pytest.approx(want, abs=1e-6)


def test_notebook_modulate_freq():
    env = [L.s2o_adsr_x16_lane(0.0, 10.0, 0.0, 10.0, n, 30) for n in range(12)]
    got = [L.s2o_modulate_freq(100.0, e, 1.0) for e in env]
    want = [200.0, 186.6066, 174.1101, 162.4505, 151.5717, 141.4214, 131.9508, 123.1144, 114.8698,
            107.1773, 100.0, 100.0]
    assert got == pytest.approx(want, rel=2e-6)


# ---- derived known answers (computed from the reference definitions) ---------------------------

def test_units_derived():
    assert L.s2o_ms_as_samples(100.0, 48000) == 4800.0
    assert L.s2o_ms_as_samples(200.0, 48000) == 9600.0
    assert L.s2o_hz_as_samples(440.0, 48000) == f32(48000.0) / f32(440.0)
    assert L.s2o_note_to_pitch(69) == 440.0
    assert L.s2o_note_to_pitch(81) == 880.0
    assert L.s2o_note_to_pitch(57) == 220.0


def test_one_pole_coefficient_derived():
    # *derived*, independently in numpy: t = ((-2*pi)*200)/48000 in f32 steps, k = RN32(exp(t))
    import math
    t = f32(f32(f32(-2.0) * f32(math.pi)) * f32(200.0)) / f32(48000.0)
    k = L.s2o_lpf_coeff(200.0, 48000)
    assert f32(k) == f32(math.exp(float(t)))
    assert k == pytest.approx(0.9741598, abs=3e-8)
    assert f32(1.0) - f32(k) == pytest.approx(0.025840223, abs=1e-9)
    last = np.zeros(1, dtype=np.float32)
    y = L.s2o_lpf_process(last.ctypes.data, 48000, 200.0, 1.0)
    assert y == last[0] == f32(1.0) - f32(k)


def test_noise_range_and_fast_form_is_exact():
    """value/65535*2-1 spans exactly [-1, 1]; the kernel's division-free form equals it for every
    possible 16-bit hash value (seed 0: the low 16 bits of n*K are a bijection of n's low 16)."""
    seen = set()
    lo, hi = 1.0, -1.0
    for n in range(65536):
        a = L.s2o_hash_noise(0, float(n))
        b = L.s2o_noise_fast_form(0, n)
        assert np.float32(a).tobytes() == np.float32(b).tobytes()
        seen.add(L.s2o_hash_word(0, n) & 0xFFFF)
        lo, hi = min(lo, a), max(hi, a)
    assert len(seen) == 65536
    assert lo == -1.0 and hi == 1.0


def test_noise_differs_from_reciprocal_multiply():
    """*derived* (SURVEY 8c): v * (1/65535) differs from the IEEE quotient at 512 of 65,536 inputs and
    the final noise sample at 191 of them — the reason the kernel may not use a plain reciprocal."""
    v = np.arange(65536, dtype=np.float32)
    q = v / np.float32(65535.0)
    r = v * (np.float32(1.0) / np.float32(65535.0))
    assert int(np.count_nonzero(q != r)) == 512
    two, one = np.float32(2.0), np.float32(1.0)
    assert int(np.count_nonzero((q * two - one) != (r * two - one))) == 191


def test_phased_offset_never_reaches_period():
    """RN(period * phase) < period for phase < 1: `offset % period` is a no-op on the x16 path."""
    rng = np.random.default_rng(7)
    P = rng.uniform(1.0, 4096.0, 400000).astype(np.float32)
    ph = np.nextafter(np.float32(1.0), np.float32(0.0)) - rng.integers(0, 64, 400000).astype(np.float32) * np.float32(2.0 ** -24)
    ph = np.concatenate([ph, rng.uniform(0, 1, 400000).astype(np.float32)])
    P = np.concatenate([P, P])
    x = P * ph   # one f32 rounding, same as fma(P, ph, 0)
    assert np.all(x < P)
    assert np.all(np.fmod(x, P) == x)


def test_osc_shapes():
    P = f32(100.0)
    assert L.s2o_osc_sample(1, P, 0.0, 1) == 1.0                 # saw starts at +1
    assert L.s2o_osc_sample(1, P, 0.5, 1) == pytest.approx(0.0, abs=1e-6)
    assert L.s2o_osc_sample(0, P, 0.25, 1) == 1.0                # square high half
    assert L.s2o_osc_sample(0, P, 0.5, 1) == -1.0
    assert L.s2o_osc_sample(2, P, 0.0, 1) == 1.0                 # triangle +1 -> -1 -> +1
    assert L.s2o_osc_sample(2, P, 0.5, 1) == pytest.approx(-1.0, abs=1e-6)
    assert L.s2o_osc_sample(3, P, 0.25, 1) == pytest.approx(1.0, abs=1e-6)   # sine table
    assert L.s2o_osc_sample(3, P, 0.0, 1) == 0.0


def test_accum_phase_wraps():
    p = f32(0.0)
    period = f32(48000.0) / f32(440.0)
    for _ in range(2000):
        p = L.s2o_accum_phase(p, period)
        assert 0.0 <= p < 1.0


def test_sin_table_matches_reference_data():
    """tests/golden/ref_sin_table.npy holds the reference's SIN_TABLE (s2_lib/src/try3/tables.rs:1-1026): its 1024
    decimal literals, each rounded to the nearest binary32 as tools/gen_sin_table.py reads them."""
    tab = oracle.sin_table()
    assert tab.shape == (1024,)
    assert tab[0] == 0.0
    assert tab.view(np.uint32)[512] == 0xB3BBBD2E    # -8.742278e-08, not 0 (tables.rs:514)
    want = np.load(pathlib.Path(__file__).resolve().parent / "golden" / "ref_sin_table.npy")
    assert want.dtype == np.float32 and want.tobytes() == tab.tobytes()


def test_sin_table_copies_identical():
    root = pathlib.Path(__file__).resolve().parent.parent
    a = (root / "oracle" / "sin_table_bits.inc").read_text()
    b = (root / "synth2_b200" / "csrc" / "sin_table_bits.inc").read_text()
    assert a == b


# ---- x16 vs scalar divergences (SURVEY 8a) --------------------------------------------------

def test_x16_adds_gain_scalar_multiplies():
    cfg = oracle.default_config()
    st = np.zeros(1, dtype=oracle.LAYER_STATE)
    out16 = np.zeros(16, dtype=np.float32)
    L.s2o_process_layer_x16(cfg.ctypes.data, st.ctypes.data, 440.0, 48000, 4800, NONE, out16.ctypes.data)
    st2 = np.zeros(1, dtype=oracle.LAYER_STATE)
    sc = L.s2o_process_layer(cfg.ctypes.data, st2.ctypes.data, 440.0, 48000, 4800, NONE)
    # first sample: saw(phase 0) = 1; x16 input = (1 + 1) + (nz + 0), scalar input = 1*1 + nz*0
    assert out16[0] != sc


def test_x16_release_waits_for_sustain_scalar_does_not():
    # release during attack: x16 keeps attacking (release clamped to A+D), scalar releases at once
    a16 = L.s2o_adsr_x16_lane(100.0, 100.0, 0.5, 100.0, 60, 50)
    asc = L.s2o_adsr_scalar(100.0, 100.0, 0.5, 100.0, 60, 50)
    assert a16 == pytest.approx(0.6, abs=1e-6)
    assert asc == pytest.approx(0.5 * (1 - 10 / 100), abs=1e-6)


def test_buf_simd_splits_x16_and_tail():
    cfg = oracle.default_config()
    st = np.zeros(1, dtype=oracle.LAYER_STATE)
    buf = np.zeros(37, dtype=np.float32)
    assert L.s2o_process_layer_buf_simd(cfg.ctypes.data, st.ctypes.data, 440.0, 48000, 0, NONE, buf.ctypes.data, 37) == 0
    st2 = np.zeros(1, dtype=oracle.LAYER_STATE)
    a = np.zeros(16, dtype=np.float32)
    b = np.zeros(16, dtype=np.float32)
    L.s2o_process_layer_x16(cfg.ctypes.data, st2.ctypes.data, 440.0, 48000, 0, NONE, a.ctypes.data)
    L.s2o_process_layer_x16(cfg.ctypes.data, st2.ctypes.data, 440.0, 48000, 16, NONE, b.ctypes.data)
    tail = [L.s2o_process_layer(cfg.ctypes.data, st2.ctypes.data, 440.0, 48000, 32 + i, NONE) for i in range(5)]
    assert buf[:16].tobytes() == a.tobytes() and buf[16:32].tobytes() == b.tobytes()
    assert buf[32:].tolist() == tail
    assert st.tobytes() == st2.tobytes()


def test_buf_simd_overflow_is_an_error():
    cfg = oracle.default_config()
    st = np.zeros(1, dtype=oracle.LAYER_STATE)
    buf = np.zeros(32, dtype=np.float32)
    rc = L.s2o_process_layer_buf_simd(cfg.ctypes.data, st.ctypes.data, 440.0, 48000, 0xFFFFFFF0, NONE, buf.ctypes.data, 32)
    assert rc == -1   # the reference panics: process.rs:36


# ---- Synth (synth.rs) ---------------------------------------------------------------------

def test_synth_voice_allocation_and_stealing():
    s = oracle.OracleSynth()
    buf = np.zeros(16, dtype=np.float32)
    for i in range(8):
        s.note_on(40 + i)
        s.sample(buf, 48000)           # voice i is now (8 - i) * 16 frames old at the end
    used = [s.voice_info(k) for k in range(8)]
    assert [u[1] for u in used] == list(range(40, 48))      # free slots were taken in index order
    s.note_on(99)                      # all busy: steal the oldest = slot 0
    assert s.voice_info(0)[1] == 99 and s.voice_info(0)[2] == 0
    s.note_off(41)
    assert s.voice_info(1)[3] == s.voice_info(1)[2]         # release = current offset
    # a second note_off for the same note finds no active voice: nothing changes (synth.rs:73)
    before = s.voice_info(1)
    assert s.note_off(41) is False
    assert s.voice_info(1)[:4] == before[:4]


def test_synth_silence_and_overwrite():
    s = oracle.OracleSynth()
    buf = np.full(40, 7.0, dtype=np.float32)
    s.sample(buf, 48000)
    assert np.all(buf == 0.0)          # overwritten, not accumulated (synth.rs:201-202)


def test_synth_mix_is_sum_in_voice_order():
    s = oracle.OracleSynth()
    s.note_on(60); s.note_on(64); s.note_on(67)
    buf = np.zeros(64, dtype=np.float32)
    s.sample(buf, 48000)
    cfg = oracle.default_config()
    acc = np.zeros(64, dtype=np.float32)
    for note in (60, 64, 67):
        st = np.zeros(1, dtype=oracle.LAYER_STATE)
        one = np.zeros(64, dtype=np.float32)
        L.s2o_process_layer_buf_simd(cfg.ctypes.data, st.ctypes.data, L.s2o_note_to_pitch(note), 48000, 0, NONE,
                                     one.ctypes.data, 64)
        acc = acc + one
    assert buf.tobytes() == acc.tobytes()


def test_bank_render_equals_per_voice_calls_and_carries_state():
    from synth2_b200 import bankgen
    b = bankgen.make_bank(5, 400, kinds=(0, 1, 2, 3))
    st = oracle.bank_init_states(b)
    a1, bus1 = oracle.bank_render(b, st, 48000, 0, 144)
    a2, bus2 = oracle.bank_render(b, st, 48000, 0, 256)
    st_once = oracle.bank_init_states(b)
    whole, bus = oracle.bank_render(b, st_once, 48000, 0, 400)
    assert np.concatenate([a1, a2], axis=1).tobytes() == whole.tobytes()   # 144 and 400 are multiples of 16
    assert np.concatenate([bus1, bus2]).tobytes() == bus.tobytes()
    assert st.tobytes() == st_once.tobytes()
    assert np.all(st["frame_offset"] == 400)
    # multi-threaded baseline mode renders the same voices
    st_mt = oracle.bank_init_states(b)
    mt, _ = oracle.bank_render(b, st_mt, 48000, 0, 400, nthreads=3)
    assert mt.tobytes() == whole.tobytes()


# ---- the rest of dsp_filters.rs (SURVEY 8f row 4): derived known answers -------------------------

def _dsp_filter_f64(kind, sr, freq, dq, x):
    """Independent binary64 restatement of dsp_filters.rs:12-230 (same formulas, numpy doubles)."""
    th = 2.0 * np.pi * freq / sr
    y = np.zeros_like(x, dtype=np.float64)
    x1 = x2 = y1 = y2 = 0.0
    if kind in ("lp2", "hp2", "bp2"):
        if kind == "bp2":
            tn = np.tan(th / (2.0 * dq))
            beta = 0.5 * (1 - tn) / (1 + tn)
            alpha = (0.5 - beta) / 2.0
        else:
            beta = 0.5 * (1 - dq / 2 * np.sin(th)) / (1 + dq / 2 * np.sin(th))
        gamma = (0.5 + beta) * np.cos(th)
        if kind == "lp2":
            alpha = (0.5 + beta - gamma) / 4.0
        if kind == "hp2":
            alpha = (0.5 + beta + gamma) / 4.0
        for i, v in enumerate(x):
            s = {"lp2": v + 2 * x1 + x2, "hp2": v - 2 * x1 + x2, "bp2": v - x2}[kind]
            out = 2.0 * (alpha * s + gamma * y1 - beta * y2)
            x2, x1, y2, y1 = x1, v, y1, out
            y[i] = out
    else:
        gamma = np.cos(th) / (1 + np.sin(th))
        alpha = (1 + gamma) / 2 if kind == "hp1" else (1 - gamma) / 2
        for i, v in enumerate(x):
            out = alpha * ((v - x1) if kind == "hp1" else (v + x1)) + gamma * y1
            x1, y1 = v, out
            y[i] = out
    return y


@pytest.mark.parametrize("kind,freq,dq", [("lp2", 1000.0, 0.7), ("hp2", 1000.0, 0.7), ("hp2", 4000.0, 1.414),
                                          ("bp2", 1500.0, 3.0), ("bp2", 3000.0, 0.8), ("lp1", 800.0, 0.0), ("hp1", 800.0, 0.0)])
def test_dsp_filters_match_a_binary64_restatement(kind, freq, dq):
    L = oracle.lib()
    rng = np.random.default_rng(5)
    x = np.concatenate([np.ones(256), rng.uniform(-1, 1, 768)]).astype(np.float32)
    st = np.zeros(1, dtype=oracle.LAYER_STATE)
    got = np.zeros(x.size, dtype=np.float32)
    for i, v in enumerate(x):
        if kind == "lp2":
            got[i] = L.s2o_biquad_lp_process(oracle._p(st), 48000, freq, dq, float(v))
        elif kind == "hp2":
            got[i] = L.s2o_biquad_hp_process(oracle._p(st), 48000, freq, dq, float(v))
        elif kind == "bp2":
            got[i] = L.s2o_biquad_bp_process(oracle._p(st), 48000, freq, dq, float(v))
        else:
            got[i] = L.s2o_first_order_process(oracle._p(st), 48000, freq, 1 if kind == "hp1" else 0, float(v))
    ref = _dsp_filter_f64(kind, 48000.0, freq, dq, x.astype(np.float64))
    assert np.max(np.abs(got - ref)) < 2e-4
    # the responses the names promise: DC passes a low-pass, is blocked by a high-pass and a band-pass
    dc = got[200:256].mean()
    assert abs(dc - (1.0 if kind in ("lp2", "lp1") else 0.0)) < 2e-3


def test_host_tuned_baseline_build_gives_the_same_bits():
    """bench.py times the CPU baseline on `make -C oracle native` (-O3 -march=native): same source, contraction
    off, no fast-math — it must render exactly what the portable build renders."""
    from synth2_b200 import bankgen
    v = bankgen.make_bank(24, 4096, kinds=(0, 1, 2, 3), mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    outs = []
    so, handle = oracle.SO, oracle._lib
    try:
        for native in (False, True):
            if native:
                flags = oracle.use_native_build()
                if "native" not in flags:
                    pytest.skip("no compiler for the host-tuned build")
            for fk in (0, 1):
                st = oracle.bank_init_states(v)
                o, b = oracle.bank_render(v, st, 48000, fk, 1000)
                outs.append((o.tobytes(), b.tobytes(), st.tobytes()))
    finally:
        oracle.SO, oracle._lib = so, handle
    assert outs[0] == outs[2] and outs[1] == outs[3]


# ---- one whole x16 block, restated independently in numpy float32 ------------------------------------------

def _libm_f32(name):
    import ctypes
    import ctypes.util
    fn = getattr(ctypes.CDLL(ctypes.util.find_library("m")), name)
    fn.restype = ctypes.c_float
    return fn


def _x16_block_numpy(cfg, state, pitch, sr, offset, release):
    """process_layer_x16 (process.rs:88-99, 137-174, 306-379) for the saw oscillator and the one-pole low-pass,
    written from the Rust source with numpy float32 vectors — every operation a separately rounded binary32
    operation, in the source's order — and NOT from oracle/s2_oracle.c.  Transcendentals are libm's (the oracle's
    stand-in for sleef `pow` and Rust's `exp`).  Returns the 16 samples and advances `state` (phase, has_phase, last)."""
    import ctypes
    powf, expf = _libm_f32("powf"), _libm_f32("expf")
    powf.argtypes = [ctypes.c_float, ctypes.c_float]
    expf.argtypes = [ctypes.c_float]
    F = np.float32
    srf = F(sr)

    def ms(x):                                            # units.rs:44-53
        return F(srf * F(F(x) / F(1000.0)))

    def adsr(env, offs):                                  # old/simdtest.rs:270-330
        A, D, S, R = ms(env["attack"]), ms(env["decay"]), F(env["sustain"]), ms(env["release"])
        x = offs.astype(np.float32)
        sus_off = F(A + D)
        rel = np.float32(np.uint32(release)) if release != NONE else F(np.uint32(0xFFFFFFFF))
        rel = np.maximum(rel, sus_off)
        end = F(rel + R)
        in_a = x < A
        in_d = ~in_a & (x < sus_off)
        in_s = ~in_a & ~in_d & (x < rel)
        in_r = ~in_a & ~in_d & ~in_s & (x < end)
        with np.errstate(divide="ignore", invalid="ignore"):
            line = lambda rise, run, xx, y0: (F(F(rise) / F(run)) * xx).astype(np.float32) + F(y0)   # never fused (:247-261)
            a_s = line(1.0, A, x, 0.0)
            d_s = line(F(S - F(1.0)), D, (x - A).astype(np.float32), 1.0)
            r_s = line(F(-S), R, (x - rel).astype(np.float32), S)
        out = np.zeros(16, np.float32)
        out = np.where(in_a, a_s, out)
        out = np.where(in_d, d_s, out)
        out = np.where(in_s, S, out)
        out = np.where(in_r, r_s, out)
        return out.astype(np.float32)                     # in_end selects 0

    offs = np.arange(offset, offset + 16, dtype=np.uint32)
    gains = adsr(cfg["amp_env"], offs)
    mods = adsr(cfg["mod_env"], offs)

    def modulate(freq, amount):                           # process.rs:231-250
        e = (mods * F(amount)).astype(np.float32)
        return np.array([F(F(powf(2.0, float(v))) * F(freq)) for v in e], dtype=np.float32)

    osc_f = modulate(pitch, cfg["mod_env_to_osc_freq"])
    lpf_f = modulate(cfg["lpf_freq"], cfg["mod_env_to_lpf_freq"])
    periods = (srf / osc_f).astype(np.float32)            # units.rs:32-41
    # accum_phase_x16 (oscillators.rs:389-400): phases of the 16 frames, then the carried one
    ph = F(state["phase"]) if state["has_phase"] else F(0.0)          # process.rs:316 unwrap_or(0)
    phases = np.zeros(16, np.float32)
    acc = ph
    for i in range(16):
        phases[i] = acc
        acc = F(np.fmod(F(acc + F(F(1.0) / periods[i])), F(1.0)))      # (phase + 1/period) % 1.0
    state["phase"], state["has_phase"] = acc, 1
    # phased_offset_x16 with feature "fma": period.mul_add(phase, 0) (oscillators.rs:217-239), then % period (:105)
    x = np.array([F(np.float64(periods[i]) * np.float64(phases[i])) for i in range(16)], dtype=np.float32)   # exact product, one rounding
    x = np.fmod(x, periods).astype(np.float32)
    # saw: line_y_value_with_y_offset_x16(-2, period, x, 1) with fma (math.rs:27-40): slope.mul_add(x, 1)
    slope = (F(-2.0) / periods).astype(np.float32)
    saw = np.array([F(np.float64(slope[i]) * np.float64(x[i]) + 1.0) for i in range(16)], dtype=np.float32)
    osc = (saw + F(cfg["osc_gain"])).astype(np.float32)   # ADDED on the x16 path (process.rs:341-345)
    # hash noise (hashnoise.rs:33-68) at offsets cast u32 -> f32 -> u32
    seed = np.uint32(state["noise_seed"])
    rot = np.uint32((int(seed) << 5 | int(seed) >> 27) & 0xFFFFFFFF)
    o32 = offs.astype(np.float32).astype(np.uint32)
    h = ((rot ^ o32).astype(np.uint64) * np.uint64(0x9E3779B9)) & np.uint64(0xFFFFFFFF)
    v = (h & np.uint64(0xFFFF)).astype(np.float32)
    nz = ((v / F(65535.0)).astype(np.float32) * F(2.0) - F(1.0)).astype(np.float32)
    nz = (nz + F(cfg["noise"])).astype(np.float32)
    u = (osc + nz).astype(np.float32)
    # one-pole per frame (filters.rs:15-34): k = exp(-2 pi f / sr); y = (1 - k).mul_add(x, k * last)
    out = np.zeros(16, np.float32)
    last = F(state["lpf_last"])
    for i in range(16):
        t = F(F(F(F(-2.0) * F(np.pi)) * lpf_f[i]) / srf)
        k = F(expf(float(t)))
        a0 = F(F(1.0) - k)
        last = F(np.float64(a0) * np.float64(u[i]) + np.float64(F(k * last)))       # fma: exact product + rounded k*last, one rounding
        out[i] = last
    state["lpf_last"] = last
    return (out * gains).astype(np.float32)


@pytest.mark.parametrize("release", [NONE, 4800])
def test_whole_x16_blocks_match_an_independent_numpy_restatement(release):
    """*derived*: the default patch (saw, one-pole, mod envelope opening the cutoff by 10 octaves; synth.rs:125-152)
    rendered block by block through attack, decay, the cutoff sweep, sustain and release — the oracle's
    s2o_process_layer_x16 against a restatement of process.rs written in numpy float32, bit for bit."""
    cfg = oracle.default_config()
    c = cfg[0]
    assert c["osc_kind"] == 1 and c["filter_kind"] == 0
    pitch, sr = 440.0, 48000
    st_o = np.zeros(1, dtype=oracle.LAYER_STATE)
    st_n = {"phase": np.float32(0), "has_phase": 0, "lpf_last": np.float32(0), "noise_seed": 0}
    cfg_n = {"osc_gain": c["osc_gain"], "noise": c["noise"], "lpf_freq": c["lpf_freq"],
             "mod_env_to_osc_freq": c["mod_env_to_osc_freq"], "mod_env_to_lpf_freq": c["mod_env_to_lpf_freq"],
             "amp_env": {"attack": c["amp_env"]["attack_ms"], "decay": c["amp_env"]["decay_ms"],
                         "sustain": c["amp_env"]["sustain"], "release": c["amp_env"]["release_ms"]},
             "mod_env": {"attack": c["mod_env"]["attack_ms"], "decay": c["mod_env"]["decay_ms"],
                         "sustain": c["mod_env"]["sustain"], "release": c["mod_env"]["release_ms"]}}
    out_o = np.zeros(16, dtype=np.float32)
    blocks = list(range(0, 12000, 16))                    # attack, decay and the whole 200 ms sweep, sustain, release
    for off in blocks:
        L.s2o_process_layer_x16(cfg.ctypes.data, st_o.ctypes.data, pitch, sr, off, release, out_o.ctypes.data)
        out_n = _x16_block_numpy(cfg_n, st_n, pitch, sr, off, release)
        assert out_o.tobytes() == out_n.tobytes(), f"block at offset {off}: {out_o} vs {out_n}"
        assert np.float32(st_o["phase"][0]).tobytes() == np.float32(st_n["phase"]).tobytes()
