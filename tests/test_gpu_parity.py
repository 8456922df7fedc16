"""Parity of the CUDA path (through the C ABI) against the CPU oracle.

The bar (BASELINE.json north star): oscillator phase / indices / stage decisions bit-exact; float
output max |err| <= 1e-4 of full scale and SNR >= 90 dB over the whole render.  Wherever no
transcendental (exp / pow / sin / cos) separates the two sides the comparison is bit-for-bit.
"""
import numpy as np
import pytest

import oracle
import synth2_b200 as s2
from busref import assert_bus_within_bound
from synth2_b200 import bankgen

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SR = 48000
# North-star bar: max |err| <= 1e-4 of full scale, SNR >= 90 dB.  Full scale is the larger of 1.0 and the
# peak of the reference render: the x16 path ADDS the oscillator gain (process.rs:341-345), which puts a
# +1 DC on every voice, so reference renders peak near 2-3.  (At cutoffs near 100 Hz the biquad's
# alpha = (1/2 + beta - gamma)/4 cancels catastrophically in f32: a 1-ulp difference between two libm
# cosf results moves the DC gain by ~5e-5 relative — the oracle uses glibc, the GPU rounds once from f64.)
TOL_ABS = 1e-4
TOL_SNR_DB = 90.0


def snr_db(ref, got):
    ref = ref.astype(np.float64).ravel()
    err = got.astype(np.float64).ravel() - ref
    p_err = float(np.sum(err * err))
    p_ref = float(np.sum(ref * ref))
    if p_err == 0.0:
        return np.inf
    return 10.0 * np.log10(max(p_ref, 1e-300) / p_err)


def assert_parity(ref, got, what=""):
    assert ref.shape == got.shape
    assert np.all(np.isfinite(got)), what
    err = float(np.max(np.abs(got.astype(np.float64) - ref.astype(np.float64)))) if ref.size else 0.0
    snr = snr_db(ref, got)
    full_scale = max(1.0, float(np.max(np.abs(ref)))) if ref.size else 1.0
    assert err <= TOL_ABS * full_scale, f"{what}: max|err| {err:.3e} (full scale {full_scale:.2f})"
    assert snr >= TOL_SNR_DB, f"{what}: SNR {snr:.1f} dB"
    return err, snr


def bank_for(filter_kind, n, frames, **kw):
    """Synthetic bank whose cutoff sweep suits the filter (the biquad is unstable above Nyquist)."""
    kw.setdefault("mod_to_lpf_choices", bankgen.MOD_TO_LPF_BIQUAD if filter_kind == 1 else bankgen.MOD_TO_LPF_ONE_POLE)
    return bankgen.make_bank(n, frames, **kw)


def gpu_bank_render(voices, filter_kind, frames_list, want_bus=True, sr=SR):
    """Render consecutive blocks on the GPU; returns (voice_out [V, sum frames], bus, final state)."""
    V = voices.shape[0]
    total = sum(frames_list)
    outs, buses = [], []
    with s2.VoiceBank(voices, sr, filter_kind) as bank:
        for fr in frames_list:
            stride = (fr + 3) & ~3
            vo = torch.full((V, stride), float("nan"), device="cuda", dtype=torch.float32)
            bus = torch.full((fr,), float("nan"), device="cuda", dtype=torch.float32) if want_bus else None
            bank.render(fr, vo, stride, bus)
            bank.sync()
            outs.append(vo[:, :fr].cpu().numpy())
            if want_bus:
                buses.append(bus.cpu().numpy())
        st = bank.get_state()
    out = np.concatenate(outs, axis=1) if outs else np.zeros((V, 0), np.float32)
    assert out.shape == (V, total)
    return out, (np.concatenate(buses) if want_bus else None), st


def oracle_bank_render(voices, filter_kind, frames_list, sr=SR, nthreads=8):
    st = oracle.bank_init_states(voices)
    outs, buses = [], []
    for fr in frames_list:
        o, _ = oracle.bank_render(voices, st, sr, filter_kind, fr, want_bus=False, nthreads=nthreads)
        outs.append(o)
        # bus in exact reference order = sequential f32 sum over voices
        acc = np.zeros(fr, dtype=np.float32)
        for v in range(voices.shape[0]):
            if voices["active"][v]:
                acc = acc + o[v]
        buses.append(acc)
    return np.concatenate(outs, axis=1), np.concatenate(buses), st


def assert_state_parity(st_gpu, st_ref, filter_kind, exact_phase=True):
    assert np.array_equal(st_gpu["frame_offset"], st_ref["frame_offset"])
    assert np.array_equal(st_gpu["has_phase"], st_ref["has_phase"])
    if exact_phase:
        assert st_gpu["phase"].tobytes() == st_ref["phase"].tobytes()      # bit-exact
    keys = ["lpf_last"] if filter_kind == 0 else ["x1", "x2", "y1", "y2"]
    for k in keys:
        np.testing.assert_allclose(st_gpu[k], st_ref[k], atol=TOL_ABS * 4, rtol=0)


# ------------------------------------------------------------------------------ Synth mirror

FIXTURE_EVENTS = [  # SURVEY 8d config 1: (frame, op, note)
    (0, "on", 69), (96000, "on", 57), (192000, "on", 76), (240000, "off", 69),
    (336000, "off", 57), (336000, "off", 76),
]


def run_script(synth, total, events, chunk=None):
    buf = np.zeros(total, dtype=np.float32)
    cuts = sorted({0, total, *[f for f, _, _ in events if f < total]})
    for a, b in zip(cuts[:-1], cuts[1:]):
        for f, op, note in events:
            if f == a:
                synth.note_on(note, 1.0) if op == "on" else synth.note_off(note)
        if chunk is None:
            synth.sample(buf[a:b], SR)
        else:
            for c in range(a, b, chunk):
                synth.sample(buf[c:min(b, c + chunk)], SR)
    return buf


@pytest.mark.parametrize("total", [480000, 480007])
def test_synth_fixture_config1(total):
    """BASELINE config 1: default patch, scripted notes, 10 s @ 48 kHz through Synth::sample;
    480,007 also exercises the scalar tail path (process.rs:39-48)."""
    ref = run_script(oracle.OracleSynth(), total, FIXTURE_EVENTS)
    syn = s2.Synth()
    got = run_script(syn, total, FIXTURE_EVENTS)
    err, snr = assert_parity(ref, got, "synth fixture")
    assert np.max(np.abs(ref)) > 0.1
    # voice bookkeeping mirrors the reference
    osyn = oracle.OracleSynth()
    run_script(osyn, total, FIXTURE_EVENTS)
    for slot in range(8):
        g, o = syn.voice_info(slot), osyn.voice_info(slot)
        assert g[:4] == o[:4], (slot, g, o)
        if g[0]:
            assert np.float32(g[4]["phase"]).tobytes() == np.float32(o[4]["phase"]).tobytes()
    syn.close()


def test_synth_live_chunks_of_16():
    """s2_bin feeds 16-frame chunks (main.rs:138-143); chunked and one-shot rendering agree bit-for-bit."""
    ev = [(0, "on", 60), (160, "on", 67), (480, "off", 60)]
    syn_a, syn_b = s2.Synth(), s2.Synth()
    a = run_script(syn_a, 1024, ev, chunk=16)
    b = run_script(syn_b, 1024, ev)
    assert a.tobytes() == b.tobytes()
    ref = run_script(oracle.OracleSynth(), 1024, ev, chunk=16)
    assert_parity(ref, a, "live chunks")
    syn_a.close(); syn_b.close()


def test_synth_stealing_matches_reference():
    osyn, syn = oracle.OracleSynth(), s2.Synth()
    buf_o, buf_g = np.zeros(48, np.float32), np.zeros(48, np.float32)
    for i in range(11):                       # 11 note-ons into 8 slots
        osyn.note_on(40 + i); syn.note_on(40 + i)
        osyn.sample(buf_o, SR); syn.sample(buf_g, SR)
        assert_parity(buf_o, buf_g, f"steal step {i}")
    osyn.note_off(45); syn.note_off(45)
    osyn.sample(buf_o, SR); syn.sample(buf_g, SR)
    assert_parity(buf_o, buf_g)
    for slot in range(8):
        assert syn.voice_info(slot)[:4] == osyn.voice_info(slot)[:4]
    syn.close()


def test_synth_rate_change_keeps_note_off():
    """ADVICE r1: `sample_rate` is an argument of every `Synth::sample` call (synth.rs:154-156).  A note released
    through the bank and then rendered at another rate must stay released (the bank is rebuilt from the host
    mirror, which has to carry the release offset)."""
    osyn, syn = oracle.OracleSynth(), s2.Synth()
    a_o, a_g = np.zeros(4800, np.float32), np.zeros(4800, np.float32)
    osyn.note_on(57); syn.note_on(57)
    osyn.note_on(64); syn.note_on(64)
    osyn.sample(a_o, 48000); syn.sample(a_g, 48000)
    assert_parity(a_o, a_g, "before the note_off")
    osyn.note_off(57); syn.note_off(57)          # an uploaded voice: goes straight to the bank
    osyn.sample(a_o, 48000); syn.sample(a_g, 48000)
    assert_parity(a_o, a_g, "after the note_off")
    b_o, b_g = np.zeros(9600, np.float32), np.zeros(9600, np.float32)
    osyn.sample(b_o, 44100); syn.sample(b_g, 44100)      # rate change: the bank is rebuilt
    assert_parity(b_o, b_g, "after the rate change")
    for slot in range(8):
        assert syn.voice_info(slot)[:4] == osyn.voice_info(slot)[:4]
    # the released voice really is in its release: the mix decays below the level of the held note alone
    assert np.max(np.abs(b_g[-480:])) < np.max(np.abs(a_g[:480])) + 1.0
    syn.close()


def test_synth_filter_kind_change_after_the_notes_ended():
    """ADVICE r1: the filter kind may change once every voice's amp envelope has ended, not only before the
    first note ever played; while a note still sounds it is refused."""
    syn = s2.Synth()
    buf = np.zeros(4800, np.float32)
    syn.note_on(60)
    syn.sample(buf, SR)
    pat = s2.patch.default_patch()
    pat.record["filter_kind"][0] = s2.FILTER_BIQUAD_LP
    pat.record["voice"]["mod_env_to_lpf_freq"][0] = 1.0
    with pytest.raises(s2.S2Error):
        syn.set_patch(pat)                      # still sounding
    syn.note_off(60)
    for _ in range(6):                          # A + D + R = 300 ms = 14,400 frames
        syn.sample(buf, SR)
    syn.set_patch(pat)                          # silent now: allowed
    syn.note_on(62)
    syn.sample(buf, SR)
    assert np.all(np.isfinite(buf)) and np.max(np.abs(buf)) > 0.0
    syn.close()


def test_damping_must_be_positive_for_second_order_filters():
    v = bankgen.make_bank(4, 64)
    v["damping"][2] = 0.0
    for fk in (1, 2, 3):
        with pytest.raises(s2.S2Error):
            s2.VoiceBank(v, SR, fk)
    s2.VoiceBank(v, SR, 0).close()              # the one-pole does not read it


def test_offset_bound_is_recomputed_before_failing():
    """ADVICE r1: the overflow guard is a bound that only grows; voices restarted since then must not trip it."""
    v = bankgen.make_bank(2, 64)
    v["frame_offset"] = 0xFFFFFF00
    v["release_offset"] = s2.NO_RELEASE
    with s2.VoiceBank(v, SR, 0) as bank:
        out = torch.zeros((2, 128), device="cuda")
        bank.render(128, out, 128, None)         # offsets now 0xFFFFFF80
        fresh = bankgen.make_bank(2, 64)
        for i in range(2):
            bank.set_voice(i, fresh[i:i + 1])    # both restarted at offset 0
        bank.render(128, out, 128, None)         # 0xFFFFFF80 + 128 would have tripped the stale bound
        bank.sync()
        assert np.all(bank.get_state()["frame_offset"] == 128)
        v2 = bankgen.make_bank(1, 64)
        v2["frame_offset"] = 0xFFFFFFF0
        bank.set_voice(0, v2)
        with pytest.raises(s2.S2Error):
            bank.render(128, out, 128, None)     # a real overflow still fails (process.rs:36)


def test_reduce_bus_single_rank():
    """s2_bank_reduce_bus (SURVEY 8b) on a one-rank communicator: the reduce is the identity, through real NCCL."""
    from synth2_b200.shard import MasterBus
    v = bankgen.make_bank(96, 4096)
    with s2.VoiceBank(v, SR, 0) as bank:
        bank.set_pipeline(2)
        bus = torch.zeros(4096, device="cuda")
        master = torch.full((4096,), float("nan"), device="cuda")
        bank.render(4096, None, 0, bus)
        with MasterBus(0, 1, 0) as comm:
            comm.reduce(bank, bus, master, root=0, stream=torch.cuda.current_stream())
            torch.cuda.synchronize()
        assert torch.equal(bus, master)
        assert float(bus.abs().max()) > 0.0


def test_synth_silence_overwrites():
    syn = s2.Synth()
    buf = np.full(100, 3.0, np.float32)
    syn.sample(buf, SR)
    assert np.all(buf == 0.0)
    syn.close()


# ------------------------------------------------------------------------------ voice banks

def test_bank_config2_saw_square_one_pole():
    """BASELINE config 2: 1,024 saw/square voices + one-pole low-pass, 4,096-frame buffers, carried state."""
    frames = [4096, 4096, 4096]
    v = bankgen.make_bank(1024, sum(frames))
    ref, rbus, rst = oracle_bank_render(v, 0, frames)
    got, gbus, gst = gpu_bank_render(v, 0, frames)
    assert_parity(ref, got, "config 2 voices")
    assert_state_parity(gst, rst, 0)
    # bus: per-warp trees, then the reduction tree -> within their error bound of the exact sum of the same rows
    off = 0
    for fr in frames:
        assert_bus_within_bound(gbus[off:off + fr], got[:, off:off + fr], v.shape[0], "default", f"block at {off}")
        off += fr
    scale = max(1.0, float(np.max(np.abs(rbus))))
    assert float(np.max(np.abs(gbus - rbus))) <= TOL_ABS * scale
    assert snr_db(rbus, gbus) >= TOL_SNR_DB


@pytest.mark.parametrize("filter_kind", [0, 1])
def test_bank_all_kinds_noise_gain(filter_kind):
    frames = [2048, 1008]
    v = bank_for(filter_kind, 200, sum(frames), kinds=(0, 1, 2, 3))   # 200: ragged last warp
    rng = np.random.default_rng(3)
    v["osc_gain"] = rng.uniform(0, 1, 200).astype(np.float32)
    v["noise_amt"] = rng.uniform(0, 1, 200).astype(np.float32)
    ref, rbus, rst = oracle_bank_render(v, filter_kind, frames)
    got, gbus, gst = gpu_bank_render(v, filter_kind, frames)
    assert_parity(ref, got, f"kinds filter {filter_kind}")
    assert_state_parity(gst, rst, filter_kind)


@pytest.mark.parametrize("kind", [0, 1, 2, 3])
def test_waveform_and_noise_bit_exact(kind):
    """With the filter and envelope made transparent (k = exp(-huge) = 0 -> y = u exactly; A = D = 0,
    S = 1 -> g = 1) the output is (osc + gain) + (noise + amt): every bit must match, for all
    65,536 values of the 16-bit noise hash."""
    n = 64
    v = bankgen.make_bank(n, 1 << 17, kinds=(kind,))
    v["lpf_freq_hz"] = 1.0e9
    v["mod_env_to_lpf_freq"] = 0.0
    v["amp_attack_ms"] = 0.0; v["amp_decay_ms"] = 0.0; v["amp_sustain"] = 1.0
    v["release_offset"] = s2.NO_RELEASE
    v["noise_seed"][: n // 2] = 0                  # seed 0: n -> hash low 16 bits is a bijection
    frames = [65536 + 16]
    ref, _, rst = oracle_bank_render(v, 0, frames)
    got, _, gst = gpu_bank_render(v, 0, frames)
    assert got.tobytes() == ref.tobytes()
    assert gst["phase"].tobytes() == rst["phase"].tobytes()


def test_phase_trace_bit_exact():
    """Oscillator phase before every frame equals the oracle's f32 recurrence bit-for-bit."""
    frames = 96000
    notes = [24, 33, 45, 57, 60, 69, 76, 88, 100, 108, 127, 0]
    v = s2.default_voice(len(notes))
    v["active"] = 1
    v["pitch_hz"] = [s2.note_to_pitch(n) for n in notes]
    v["osc_kind"] = [i % 4 for i in range(len(notes))]
    ph = torch.zeros((len(notes), frames), device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 0) as bank:
        bank.trace_phase(frames, ph)
        bank.sync()
    got = ph.cpu().numpy()
    for i, n in enumerate(notes):
        cfg = oracle.default_config()
        cfg["osc_kind"] = v["osc_kind"][i]
        _, rph, _, _ = oracle.trace_voice(cfg, float(v["pitch_hz"][i]), SR, 0, oracle.NO_RELEASE, frames)
        assert got[i].tobytes() == rph.tobytes(), f"note {n}"


def test_pitch_matches_oracle_table():
    for n in range(128):
        assert np.float32(s2.note_to_pitch(n)).tobytes() == np.float32(oracle.lib().s2o_note_to_pitch(n)).tobytes()


@pytest.mark.parametrize("filter_kind", [0, 1])
def test_modulated_pitch_and_cutoff(filter_kind):
    """mod_env -> osc freq != 0: the period moves every frame of the mod decay (general path)."""
    frames = [4800, 4800, 2400]
    v = bank_for(filter_kind, 48, sum(frames), kinds=(0, 1, 2, 3))
    v["mod_env_to_osc_freq"] = np.linspace(-2.0, 2.0, 48).astype(np.float32)
    v["mod_decay_ms"] = 150.0
    v["mod_sustain"] = 0.3
    v["mod_release_ms"] = 20.0
    v["release_offset"] = 9600
    ref, _, rst = oracle_bank_render(v, filter_kind, frames)
    got, _, gst = gpu_bank_render(v, filter_kind, frames)
    # pow() feeds the period here: phase is compared with a tolerance, not bit-for-bit (SURVEY 7 #4)
    smooth = np.isin(v["osc_kind"], (1, 2, 3))          # a square flips +-1 on a 1-ulp phase change
    assert_parity(ref[smooth], got[smooth], "modulated pitch")
    d = np.abs(gst["phase"] - rst["phase"]); d = np.minimum(d, 1.0 - d)
    assert float(d.max()) < 1e-4
    sq = ~smooth
    assert np.mean(np.abs(got[sq] - ref[sq]) > 1e-3) < 1e-3


@pytest.mark.parametrize("frames", [1, 15, 16, 17, 31, 32, 33, 47, 48, 63, 64, 65, 4101])
@pytest.mark.parametrize("nv", [1, 33])
def test_ragged_frames_and_voices(frames, nv):
    v = bankgen.make_bank(nv, 400, kinds=(1, 0, 3, 2))
    v["noise_amt"] = 0.25
    ref, rbus, rst = oracle_bank_render(v, 0, [frames, frames])
    got, gbus, gst = gpu_bank_render(v, 0, [frames, frames])
    assert_parity(ref, got, f"frames {frames} nv {nv}")
    assert_state_parity(gst, rst, 0)
    if nv <= 32:
        # a single warp adds its voices in index order from 0.0: the reference's mix order
        mix = np.zeros(2 * frames, np.float32)
        for r in got:
            mix = mix + r
        assert gbus.tobytes() == mix.tobytes()


def test_empty_render_is_a_noop():
    v = bankgen.make_bank(4, 64)
    with s2.VoiceBank(v, SR, 0) as bank:
        bank.render(0, None, 0, None)
        st = bank.get_state()
    assert np.all(st["frame_offset"] == 0) and np.all(st["has_phase"] == 0)


def test_inactive_voices_set_voice_release_voice():
    frames = 1024
    v = bankgen.make_bank(40, 4 * frames, kinds=(1, 0))
    v["release_offset"] = s2.NO_RELEASE
    v["active"][::3] = 0
    ref_v = v.copy()
    st = oracle.bank_init_states(ref_v)
    r1, _ = oracle.bank_render(ref_v, st, SR, 0, frames, want_bus=False)
    # note_on into slot 3 (was inactive), note_off slot 1
    nv = bankgen.make_bank(1, 4 * frames, first_voice=999)[0:1].copy()
    nv["release_offset"] = s2.NO_RELEASE
    ref_v[3] = nv[0]
    st[3] = np.zeros(1, dtype=st.dtype)[0]
    ref_v["release_offset"][1] = st["frame_offset"][1]
    r2, _ = oracle.bank_render(ref_v, st, SR, 0, frames, want_bus=False)

    with s2.VoiceBank(v, SR, 0) as bank:
        o1 = torch.zeros((40, frames), device="cuda"); o2 = torch.zeros((40, frames), device="cuda")
        bank.render(frames, o1)
        bank.set_voice(3, nv)
        bank.release_voice(1)
        bank.render(frames, o2)
        bank.sync()
        gst = bank.get_state()
    g1, g2 = o1.cpu().numpy(), o2.cpu().numpy()
    assert_parity(r1, g1); assert_parity(r2, g2)
    assert np.all(g1[::3] == 0.0)                         # inactive rows are written as zeros
    assert gst["frame_offset"][0] == 0                    # ... and do not advance
    assert gst["frame_offset"][1] == 2 * frames and gst["frame_offset"][3] == frames


@pytest.mark.parametrize("start", [(1 << 24) - 40, (1 << 24) + 1000, 0xFFFFFFFF - 5000])
def test_large_frame_offsets(start):
    """Offsets are converted u32 -> f32 (simdtest.rs:277-279, process.rs:347-348): exact only below 2^24."""
    v = bankgen.make_bank(8, 1000, kinds=(1, 0, 2, 3))
    v["frame_offset"] = start
    v["release_offset"] = start + 160
    v["noise_amt"] = 0.5
    frames = [304, 96]
    ref, _, rst = oracle_bank_render(v, 0, frames)
    got, _, gst = gpu_bank_render(v, 0, frames)
    assert_parity(ref, got, f"offset {start}")
    assert_state_parity(gst, rst, 0)


def test_frame_offset_overflow_is_an_error():
    v = bankgen.make_bank(2, 64)
    v["frame_offset"] = 0xFFFFFFFF - 100
    with s2.VoiceBank(v, SR, 0) as bank:
        with pytest.raises(s2.S2Error) as e:
            bank.render(128, None, 0, None)
        assert e.value.code == -4


def test_state_checkpoint_and_migrate():
    frames = 2048
    for fk in (0, 1):
        v = bank_for(fk, 96, 3 * frames, kinds=(0, 1, 2, 3))
        whole, _, st_whole = gpu_bank_render(v, fk, [frames, frames])
        with s2.VoiceBank(v, SR, fk) as a:
            o1 = torch.zeros((96, frames), device="cuda")
            a.render(frames, o1); a.sync()
            ck = a.get_state()
        with s2.VoiceBank(v, SR, fk) as b:
            b.set_state(ck)
            o2 = torch.zeros((96, frames), device="cuda")
            b.render(frames, o2); b.sync()
            st_b = b.get_state()
        both = np.concatenate([o1.cpu().numpy(), o2.cpu().numpy()], axis=1)
        assert both.tobytes() == whole.tobytes()
        assert st_b.tobytes() == st_whole.tobytes()


def test_split_invariance_bitwise():
    """Rendering T frames in one call or in pieces (multiples of 16) gives identical bits and state."""
    for fk in (0, 1):
        v = bank_for(fk, 64, 8192, kinds=(1, 0))
        a, _, sa = gpu_bank_render(v, fk, [8192])
        b, _, sb = gpu_bank_render(v, fk, [4096, 2048, 16, 2032])
        assert a.tobytes() == b.tobytes()
        assert sa.tobytes() == sb.tobytes()


@pytest.mark.parametrize("filter_kind", [0, 1, 2, 4])
def test_paths_agree_bitwise(filter_kind, monkeypatch):
    """Purity of the per-frame functions (s2_cutoff.h): the specialised paths of the render kernel — fast tiles,
    packed moving-cutoff chunks with the resting lane of a pair helping its moving partner (default) and without
    (S2_FORCE_PATH=3), one-frame-at-a-time moving-cutoff chunks (1) — and the general per-frame path
    (S2_FORCE_PATH=2) perform the same IEEE operations per frame: identical bits, including through envelope
    ramps, moving cutoffs (window-aligned and not), pitch modulation and the scalar tail."""
    frames = [4096, 4096, 2048, 1000]
    v = bank_for(1 if filter_kind else 0, 160, sum(frames), kinds=(0, 1, 2, 3))
    v["noise_amt"] = (np.arange(160) % 2) * 0.5
    v["mod_env_to_osc_freq"][::7] = 0.5
    v["mod_decay_ms"] = np.where(np.arange(160) % 3 == 0, 200.0, 83.3).astype(np.float32)
    v["mod_attack_ms"][64:] = 11.0
    v["frame_offset"][96:] = 16 * (np.arange(64) % 5)
    v["release_offset"] = 6000
    outs = {}
    for path in ("0", "1", "2", "3"):
        monkeypatch.setenv("S2_FORCE_PATH", path)
        outs[path] = gpu_bank_render(v, filter_kind, frames)
    monkeypatch.delenv("S2_FORCE_PATH")
    a = outs["2"]
    assert np.all(np.isfinite(a[0]))
    for name in ("0", "1", "3"):
        b = outs[name]
        bad = np.argwhere(a[0] != b[0])
        assert bad.size == 0, f"path {name}: first differing (voice, frame): {bad[:5].tolist()}"
        assert a[2].tobytes() == b[2].tobytes()
        assert a[1].tobytes() == b[1].tobytes()


@pytest.mark.parametrize("followers", [0.0, 0.2, 0.8, 1.0])
def test_lane_pair_layouts_agree_bitwise(followers, monkeypatch):
    """s2_bank_create pairs voices whose cutoff follows the mod envelope with voices whose cutoff rests (aligned
    lane pairs, chunk_modcut_pr); with few or many followers some voices find no partner and whole warps fall back
    to chunk_modcut_pk.  Whatever the proportion, the output is the general per-frame path's (S2_FORCE_PATH=2) bit
    for bit, in the caller's voice order, and within the bar of the oracle."""
    frames = [4096, 4096, 2048]
    n = 333                                           # ragged last warp, odd group sizes
    v = bank_for(1, n, sum(frames), kinds=(0, 1, 2))
    rng = np.random.default_rng(int(followers * 10) + 7)
    v["mod_env_to_lpf_freq"] = np.where(rng.uniform(size=n) < followers, 1.5, 0.0).astype(np.float32)
    v["active"][5::41] = 0
    outs = {}
    for path in ("0", "2"):
        monkeypatch.setenv("S2_FORCE_PATH", path)
        outs[path] = gpu_bank_render(v, 1, frames)
    monkeypatch.delenv("S2_FORCE_PATH")
    a, b = outs["0"], outs["2"]
    bad = np.argwhere(a[0] != b[0])
    assert bad.size == 0, f"first differing (voice, frame): {bad[:5].tolist()}"
    assert a[2].tobytes() == b[2].tobytes()
    ref, _, _ = oracle_bank_render(v, 1, frames)
    assert_parity(ref, a[0], f"lane pairs, {followers:.0%} followers")


@pytest.mark.parametrize("n_sub", [2, 4, 8])
def test_pipelined_sub_banks_agree_bitwise(n_sub):
    """s2_bank_set_pipeline: the same voices rendered as n_sub ranges on internal streams give the same
    bits as the single-stream bank — per-voice output, carried state, and the note-off table path."""
    frames = [4096, 4096, 2048, 1000, 4096]
    V = 1000                                   # not a multiple of 64 * n_sub
    v = bank_for(1, V, sum(frames), kinds=(0, 1, 2, 3))
    v["release_offset"] = s2.NO_RELEASE
    rel = np.full(V, s2.NO_RELEASE, dtype=np.uint32)
    rel[::3] = 5000
    rel[1::3] = 9000

    def run(pipe):
        outs, buses = [], []
        with s2.VoiceBank(v, SR, 1) as bank:
            if pipe > 1:
                bank.set_pipeline(pipe)
            for i, fr in enumerate(frames):
                if i == 1:
                    bank.set_releases(rel)
                stride = (fr + 3) & ~3
                vo = torch.full((V, stride), float("nan"), device="cuda")
                bus = torch.full((fr,), float("nan"), device="cuda")
                bank.render(fr, vo, stride, bus)
                bank.sync()
                outs.append(vo[:, :fr].cpu().numpy())
                buses.append(bus.cpu().numpy())
            return np.concatenate(outs, axis=1), np.concatenate(buses), bank.get_state()

    a = run(1)
    b = run(n_sub)
    assert np.all(np.isfinite(b[0]))
    assert a[0].tobytes() == b[0].tobytes()
    assert a[2].tobytes() == b[2].tobytes()
    assert a[1].tobytes() == b[1].tobytes()    # same warps, same fixed reduction tree
    # and against the oracle, with the note-off table applied from the second block on
    ref_v = v.copy()
    st = oracle.bank_init_states(ref_v)
    o0, _ = oracle.bank_render(ref_v, st, SR, 1, frames[0], want_bus=False, nthreads=8)
    ref_v["release_offset"] = rel
    o1, _ = oracle.bank_render(ref_v, st, SR, 1, frames[1], want_bus=False, nthreads=8)
    assert_parity(np.concatenate([o0, o1], axis=1), b[0][:, :frames[0] + frames[1]], "pipelined vs oracle")


def test_note_off_table_survives_a_pipeline_change():
    """A note-off table staged for the next pipelined render (the render kernels of the ranges apply it in their
    prologues) is not lost when the number of ranges changes first, or when the bank goes back to one stream."""
    frames = [2048, 4096]
    V = 500
    v = bank_for(1, V, sum(frames), kinds=(0, 1))
    v["release_offset"] = s2.NO_RELEASE
    rel = np.full(V, s2.NO_RELEASE, dtype=np.uint32)
    rel[::2] = 3000

    def run(first, second):
        with s2.VoiceBank(v, SR, 1) as bank:
            if first > 1:
                bank.set_pipeline(first)
            outs = []
            for i, fr in enumerate(frames):
                if i == 1:
                    bank.set_releases(rel)
                    if second != first:
                        bank.set_pipeline(second)
                vo = torch.full((V, fr), float("nan"), device="cuda")
                bank.render(fr, vo, fr, None)
                bank.sync()
                outs.append(vo.cpu().numpy())
            return np.concatenate(outs, axis=1), bank.get_state()

    a = run(1, 1)
    for first, second in ((4, 4), (4, 2), (4, 1), (1, 4)):
        b = run(first, second)
        assert a[0].tobytes() == b[0].tobytes(), (first, second)
        assert a[1].tobytes() == b[1].tobytes(), (first, second)


def test_pipelined_back_to_back_without_sync():
    """Many blocks enqueued without a host sync in between (the bench shape), joined at the end."""
    V, T, N = 4096, 1024, 24
    v = bank_for(1, V, N * T)
    whole, _, st_ref = gpu_bank_render(v, 1, [T] * N, want_bus=False)
    ring = [torch.empty((V, T), device="cuda") for _ in range(N)]
    host_bus = [torch.empty(T).pin_memory() for _ in range(N)]
    with s2.VoiceBank(v, SR, 1, stream=torch.cuda.current_stream()) as bank:
        bank.set_pipeline(4)
        for i in range(N):
            bank.render_bus_host_async(T, host_bus[i], ring[i], T)
        bank.join(torch.cuda.current_stream())
        torch.cuda.current_stream().synchronize()
        st = bank.get_state()
    got = torch.cat(ring, dim=1).cpu().numpy()
    assert got.tobytes() == whole.tobytes()
    assert st.tobytes() == st_ref.tobytes()
    for i in range(N):
        assert_bus_within_bound(host_bus[i].numpy(), ring[i], V, "pipelined", f"block {i}")


@pytest.mark.parametrize("seed", range(12))
def test_random_banks_against_oracle(seed):
    """Seeded random patches, offsets, release points, block splits, lane layouts and pipelining."""
    rng = np.random.default_rng(1000 + seed)
    fk = int(rng.integers(0, 2))
    V = int(rng.choice([1, 7, 32, 33, 96, 130, 257]))
    frames = [int(x) for x in rng.choice([16, 48, 250, 512, 1000, 2048, 3001], size=int(rng.integers(1, 4)))]
    v = s2.default_voice(V)
    v["active"] = (rng.random(V) > 0.1).astype(np.uint32)
    v["osc_kind"] = rng.integers(0, 4, V)
    v["noise_seed"] = rng.integers(0, 2 ** 32, V, dtype=np.uint64).astype(np.uint32)
    v["pitch_hz"] = [s2.note_to_pitch(int(n)) for n in rng.integers(12, 120, V)]
    v["osc_gain"] = rng.choice([0.0, 0.5, 1.0], V).astype(np.float32)
    v["noise_amt"] = rng.choice([0.0, 0.0, 0.3, 1.0], V).astype(np.float32)
    v["lpf_freq_hz"] = np.exp(rng.uniform(np.log(150.0), np.log(6000.0), V)).astype(np.float32)
    v["damping"] = rng.uniform(0.3, 1.414, V).astype(np.float32)
    for env, lo in (("amp", 0.0), ("mod", 0.0)):
        v[f"{env}_attack_ms"] = rng.choice([0.0, 1.0, 7.3, 40.0], V).astype(np.float32)
        v[f"{env}_decay_ms"] = rng.choice([0.0, 3.0, 25.0, 90.0], V).astype(np.float32)
        v[f"{env}_sustain"] = rng.uniform(lo, 1.0, V).astype(np.float32)
        v[f"{env}_release_ms"] = rng.choice([0.0, 2.0, 30.0], V).astype(np.float32)
    v["mod_env_to_lpf_freq"] = rng.choice([0.0, 0.0, 1.0, -1.5], V).astype(np.float32) if fk else \
        rng.choice([0.0, 10.0, -3.0, 4.5], V).astype(np.float32)
    v["mod_env_to_osc_freq"] = 0.0
    start = int(rng.choice([0, 0, 16, 4800, (1 << 24) - 700]))
    v["frame_offset"] = start + 16 * rng.integers(0, 4, V)
    rel = v["frame_offset"] + rng.integers(0, sum(frames) + 200, V)
    v["release_offset"] = np.where(rng.random(V) < 0.3, s2.NO_RELEASE, rel).astype(np.uint32)
    ref, rbus, rst = oracle_bank_render(v, fk, frames)
    mode = seed % 4
    env = {1: ("S2_FORCE_PATH", "1"), 2: ("S2_FORCE_PATH", "2")}.get(mode)
    import os
    if env:
        os.environ[env[0]] = env[1]
    try:
        if mode == 3:
            outs = []
            with s2.VoiceBank(v, SR, fk) as bank:
                bank.set_pipeline(3)
                for fr in frames:
                    stride = (fr + 3) & ~3
                    vo = torch.full((V, stride), float("nan"), device="cuda")
                    bank.render(fr, vo, stride, None)
                    bank.sync()
                    outs.append(vo[:, :fr].cpu().numpy())
                gst = bank.get_state()
            got = np.concatenate(outs, axis=1)
        else:
            got, gbus, gst = gpu_bank_render(v, fk, frames)
    finally:
        if env:
            del os.environ[env[0]]
    assert_parity(ref, got, f"fuzz seed {seed} fk {fk} V {V} frames {frames} mode {mode}")
    assert_state_parity(gst, rst, fk)


def test_errors_are_reported_not_crashes():
    v = bankgen.make_bank(4, 64)
    bad = v.copy(); bad["osc_kind"][0] = 9
    with pytest.raises(s2.S2Error):
        s2.VoiceBank(bad, SR, 0)
    bad = v.copy(); bad["pitch_hz"][1] = float("nan")
    with pytest.raises(s2.S2Error):
        s2.VoiceBank(bad, SR, 0)
    with pytest.raises(s2.S2Error):
        s2.VoiceBank(v, SR, 7)
    with s2.VoiceBank(v, SR, 0) as bank:
        buf = torch.zeros(4 * 64 + 1, device="cuda")
        with pytest.raises(s2.S2Error):            # misaligned rows
            bank.render(64, buf[1:], 64, None)
        with pytest.raises(s2.S2Error):
            bank.set_voice(10, v[0:1])


def test_whole_render_parity_config3():
    """BASELINE config 3 over the WHOLE render (north star: "over the whole render"): 65,536 voices, resonant
    biquad + ADSR, 60 s = 2,880,000 frames in 704 blocks through the pipelined path the bench times (4 voice ranges),
    the DSP state carried on the device across all of them (state.rs:8-21, synth.rs:24-30,197).  64 voice rows are
    gathered from every block — 32 spread over the bank (both kinds), 32 from the corner where the second-order
    low-pass is least forgiving in binary32 (lowest cutoff x damping among the voices whose cutoff follows the mod
    envelope) — and compared with the oracle frame by frame: final phase and offset bit-for-bit, max |err| unscaled
    and over the reference peak, SNR.

    The bar is the north star's 1e-4 of full scale / 90 dB.  Where a voice misses 1e-4 UNSCALED it is listed in the
    report (DESIGN.md section 5 holds the list of the committed run) and held to the reference's own sensitivity
    instead: the oracle's response to moving that voice's cutoff by ONE ulp.  At 100 Hz and damping 0.2 the
    binary32 direct form amplifies any last-bit difference — sleef `pow` against libm `powf` in the reference itself —
    into a few 1e-4; an error within a small multiple of that is indistinguishable from the reference's own."""
    import json, os, pathlib
    V, T, total = 65536, 4096, 2880000
    v = bank_for(1, V, total)
    even = np.linspace(0, V - 1, 32).astype(np.int64)
    score = v["lpf_freq_hz"].astype(np.float64) * v["damping"] + np.where(v["mod_env_to_lpf_freq"] != 0, 0.0, 1e9)
    corner = np.argsort(score, kind="stable")[:32]
    idx = np.unique(np.concatenate([even, corner]))
    is_corner = np.isin(idx, corner)
    sub = np.ascontiguousarray(v[idx])
    bumped = sub.copy()
    bumped["lpf_freq_hz"] = np.nextafter(sub["lpf_freq_hz"], np.float32(np.inf))
    st_ref, st_bump = oracle.bank_init_states(sub), oracle.bank_init_states(bumped)
    n = idx.size
    max_err, max_sens, peak = np.zeros(n), np.zeros(n), np.zeros(n)
    p_err, p_ref = np.zeros(n), np.zeros(n)
    ring = [torch.empty((V, T), device="cuda", dtype=torch.float32) for _ in range(2)]
    sel = torch.as_tensor(idx, device="cuda")
    stream = torch.cuda.current_stream()
    with s2.VoiceBank(v, SR, 1, stream=stream) as bank:
        bank.set_pipeline(4)
        pos, i = 0, 0
        pending = None
        while pos < total:
            fr = min(T, total - pos)
            bank.render(fr, ring[i & 1], T, None)
            bank.join(stream)
            rows = ring[i & 1].index_select(0, sel)[:, :fr].to("cpu", non_blocking=False).numpy()
            ref, _ = oracle.bank_render(sub, st_ref, SR, 1, fr, want_bus=False, nthreads=os.cpu_count() or 1)
            bmp, _ = oracle.bank_render(bumped, st_bump, SR, 1, fr, want_bus=False, nthreads=os.cpu_count() or 1)
            assert np.all(np.isfinite(rows)), f"block {i}"
            e = np.abs(rows.astype(np.float64) - ref)
            max_err = np.maximum(max_err, e.max(axis=1))
            max_sens = np.maximum(max_sens, np.abs(bmp.astype(np.float64) - ref).max(axis=1))
            peak = np.maximum(peak, np.abs(ref).max(axis=1))
            p_err += (e * e).sum(axis=1)
            p_ref += (ref.astype(np.float64) ** 2).sum(axis=1)
            pos += fr
            i += 1
        gst = bank.get_state()[idx]
    assert i == 704
    assert np.array_equal(gst["phase"].view(np.uint32), st_ref["phase"].view(np.uint32)), "final phase"
    assert np.array_equal(gst["frame_offset"], st_ref["frame_offset"]), "final offset"
    snr = 10.0 * np.log10(np.maximum(p_ref, 1e-300) / np.maximum(p_err, 1e-300))
    full_scale = max(1.0, float(peak.max()))
    over = [{"voice": int(idx[k]), "cutoff_hz": float(sub["lpf_freq_hz"][k]), "damping": float(sub["damping"][k]),
             "follows_mod_env": bool(sub["mod_env_to_lpf_freq"][k] != 0), "max_abs_err": float(max_err[k]),
             "one_ulp_of_cutoff_moves_the_reference_by": float(max_sens[k]), "snr_db": float(snr[k])}
            for k in np.argsort(-max_err) if max_err[k] > TOL_ABS]
    report = {"voices": int(n), "frames": total, "blocks": i, "phase_bit_exact": True,
              "max_abs_err_unscaled": float(max_err.max()), "ref_peak": float(peak.max()),
              "max_abs_err_over_ref_peak": float(max_err.max() / full_scale),
              "spread_sample": {"max_abs_err": float(max_err[~is_corner].max()), "min_snr_db": float(snr[~is_corner].min())},
              "corner_sample": {"max_abs_err": float(max_err[is_corner].max()), "min_snr_db": float(snr[is_corner].min()),
                                "max_one_ulp_sensitivity": float(max_sens[is_corner].max())},
              "voices_over_1e-4_unscaled": over}
    print("whole-render parity:", json.dumps(report))
    out_dir = pathlib.Path(__file__).resolve().parent.parent / "gpurun_out"
    if out_dir.is_dir():
        (out_dir / "whole_render_parity.json").write_text(json.dumps(report, indent=1) + "\n")
    for k in range(n):
        bound = max(TOL_ABS * full_scale, 4.0 * max_sens[k])
        assert max_err[k] <= bound, (f"voice {int(idx[k])} (cutoff {sub['lpf_freq_hz'][k]:.1f} Hz, damping {sub['damping'][k]:.3f}): "
                                     f"max|err| {max_err[k]:.3e} > max(1e-4 FS, 4 x one-ulp sensitivity {max_sens[k]:.3e})")
    assert float(snr[~is_corner].min()) >= TOL_SNR_DB, f"SNR of the spread sample {snr[~is_corner].min():.1f} dB"
    assert float(max_err[~is_corner].max()) <= TOL_ABS * full_scale


def test_full_size_properties_config3():
    """BASELINE config 3 shape at full width: 65,536 voices x 4,096-frame block, resonant biquad + ADSR.
    Checked through size-independent properties plus an oracle comparison of a voice sample."""
    V, T = 65536, 4096
    v = bank_for(1, V, 2880000)
    out = torch.empty((V, T), device="cuda", dtype=torch.float32)
    bus = torch.empty(T, device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 1) as bank:
        bank.render(T, out, T, bus)
        bank.sync()
        st1 = bank.get_state()
    assert bool(torch.isfinite(out).all())
    # (1) a sample of voices against the oracle
    pick = np.sort(np.random.default_rng(11).choice(V, 96, replace=False))
    ref, _, rst = oracle_bank_render(v[pick].copy(), 1, [T])
    got = out[torch.as_tensor(pick, device="cuda")].cpu().numpy()
    assert_parity(ref, got, "config 3 sample")
    assert st1["phase"][pick].tobytes() == rst["phase"].tobytes()
    # (2) the bus is the sum of the rows
    assert_bus_within_bound(bus, out, V, "default", "config 3")
    # (3) split invariance at full width: two half blocks give the same bits
    out2 = torch.empty((V, T), device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 1) as bank:
        bank.render(T // 2, out2, T, None)
        bank.render(T // 2, out2[:, T // 2:], T, None)
        bank.sync()
        st2 = bank.get_state()
    assert bool(torch.equal(out, out2))
    assert st1.tobytes() == st2.tobytes()


def test_sweep_variants_config5():
    """BASELINE config 5 (one GPU's share): the 32 x 32 x 32 cutoff / damping / detune grid of the default
    patch through the resonant low-pass.  A strided sample of variants against the oracle over the first
    notes of the render (the moving-cutoff segment, decay, sustain), then at full width: every variant
    renders exactly as it does alone (independence), and no variant blows up."""
    T = 4096
    blocks = [T, T, T, 1024]                       # 13,312 frames: past the 200 ms mod decay and the amp decay
    v = bankgen.make_sweep_bank(1, 480000)
    pick = np.arange(5, 32768, 517)                # 64 variants, all three axes move
    sub = v[pick].copy()
    ref, _, rst = oracle_bank_render(sub, 1, blocks)
    got, _, st = gpu_bank_render(sub, 1, blocks, want_bus=False)
    assert_parity(ref, got, "sweep sample")
    assert_state_parity(st, rst, 1)
    # full width, first block: the sample's rows come out bit-identical inside the 32,768-variant bank.  There
    # every warp is 32 detunes of one (cutoff, damping) pair, so the moving-cutoff chunks compute their
    # coefficients once per warp, one frame per lane (modcut_coefficients + chunk_modcut_sc<SHARED>); the 64-variant sample above took the
    # per-voice form.  Silent voices parked at another frame offset must not disturb their warp.
    idle = np.setdiff1d(np.arange(7, 32768, 32), pick)
    v["active"][idle] = 0
    v["frame_offset"][idle] = 777
    out = torch.empty((32768, T), device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 1) as bank:
        bank.set_pipeline(4)
        bank.render(T, out, T, None)
        bank.sync()
    assert bool(torch.isfinite(out).all())
    rows = out[torch.as_tensor(pick, device="cuda")].cpu().numpy()
    assert rows.tobytes() == got[:, :T].tobytes()
    assert bool((out[torch.as_tensor(idle, device="cuda")] == 0).all())
    # release at 75 % of a short render: the tail decays to silence for every variant
    short = bankgen.make_sweep_bank(1, 16384, first_variant=0, n_variants=1024)
    o, _, _ = gpu_bank_render(short, 1, [16384, 4096 + 2048], want_bus=False)
    assert np.all(o[:, 12288 + 4800:] == 0.0)      # release 100 ms = 4,800 frames after frame 12,288
    assert np.all(np.abs(o[:, 12288 + 4700]) > 0.0)


# ------------------------------------------------------------------------------ time-split (narrow banks)

def _render_blocks(voices, filter_kind, blocks, time_split, kinds_stride=None):
    V = voices.shape[0]
    outs = []
    with s2.VoiceBank(voices, SR, filter_kind) as bank:
        if time_split:
            bank.set_time_split(True)
        for fr in blocks:
            vo = torch.full((V, fr), float("nan"), device="cuda", dtype=torch.float32)
            bank.render(fr, vo, fr, None)
            bank.sync()
            outs.append(vo.cpu().numpy())
        st = bank.get_state()
        n_ts = bank.time_split_blocks
    return np.concatenate(outs, axis=1), st, n_ts


def test_time_split_config2_against_oracle():
    """BASELINE config 2 through the time-split kernels: 1,024 saw/square voices + one-pole low-pass,
    4,096-frame buffers, carried state.  Every block renders as 32 segments per voice: the first three
    (200 ms mod-envelope decay on half the voices) with per-frame filter coefficients, the rest with constant
    ones.  Phase bit-exact, output within the north-star tolerance, against the oracle and the default path."""
    V, T, N = 1024, 4096, 6
    v = bank_for(0, V, 400000)
    ref, _, rst = oracle_bank_render(v, 0, [T] * N)
    got, st, n_ts = _render_blocks(v, 0, [T] * N, True)
    assert n_ts == N
    assert_parity(ref, got, "config 2 time-split vs oracle")
    assert_state_parity(st, rst, 0)
    plain, st0, n0 = _render_blocks(v, 0, [T] * N, False)
    assert n0 == 0
    assert st["phase"].tobytes() == st0["phase"].tobytes()
    assert np.array_equal(st["frame_offset"], st0["frame_offset"])
    assert_parity(plain, got, "config 2 time-split vs default path")


def test_time_split_envelopes_kinds_and_fallbacks():
    """Every block qualifies when the cutoff ignores the mod envelope: attack / decay / release ramps then
    cross segment boundaries inside a block, and the release lands mid-block.  All four oscillators, noise
    amount, inactive voices; block lengths that are not a multiple of 1,024 fall back to the default path."""
    V = 160
    v = bank_for(0, V, 20480, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE),
                 mod_to_lpf_choices=(0.0,))
    v["noise_amt"][::3] = 0.25
    v["osc_gain"][::5] = 0.5
    v["active"][7::31] = 0
    v["release_offset"][::2] = 9000           # not a multiple of 16: note-offs land anywhere
    blocks = [4096, 2048, 1024, 4096, 1000, 3096, 8192]
    ref, _, rst = oracle_bank_render(v, 0, blocks)
    got, st, n_ts = _render_blocks(v, 0, blocks, True)
    assert n_ts == 5                          # 1000 and 3096 are not multiples of 1,024
    assert_parity(ref, got, "time-split envelopes/kinds")
    assert_state_parity(st, rst, 0)
    assert np.all(got[v["active"] == 0] == 0.0)


def test_time_split_follows_note_offs_and_mod_release():
    """Blocks in which a cutoff follows a ramping mod envelope (decay after the note-on, release after the
    note-off, stage changes mid-segment) take the per-frame-coefficient form of the time-split kernels."""
    V, T = 64, 2048
    v = bank_for(0, V, 10 * T)                # release at 15,360 = block 7.5
    v["mod_release_ms"] = 20.0
    v["mod_sustain"] = 0.6
    ref, _, rst = oracle_bank_render(v, 0, [T] * 10)
    got, st, n_ts = _render_blocks(v, 0, [T] * 10, True)
    # blocks 0-4 hold the 9,600-frame decay, block 7 the release start (and its 960-frame ramp)
    assert n_ts == 10
    assert_parity(ref, got, "time-split mod release")
    assert_state_parity(st, rst, 0)


def test_time_split_biquad_2x2_scan():
    """The second-order low-pass through the time-split kernels: the (y1, y2) state enters each segment through
    the prefix scan of the segments' 2x2 affine maps, the delayed inputs x1, x2 are recomputed from the two
    frames before the segment.  Resonant and low-cutoff voices included (the bank draws damping from
    [0.2, 1.414] and cutoffs from 100 Hz); all oscillator kinds; against the oracle and the default path."""
    V, T, N = 256, 4096, 5
    v = bank_for(1, V, 400000, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE))
    v["noise_amt"][::4] = 0.2
    v["active"][5::17] = 0
    ref, _, rst = oracle_bank_render(v, 1, [T] * N)
    got, st, n_ts = _render_blocks(v, 1, [T] * N, True)
    assert n_ts == N                          # blocks 0-2 (mod decay) with per-frame 2x2 maps
    assert_parity(ref, got, "biquad time-split vs oracle")
    assert_state_parity(st, rst, 1)
    plain, st0, _ = _render_blocks(v, 1, [T] * N, False)
    assert st["phase"].tobytes() == st0["phase"].tobytes()
    assert_parity(plain, got, "biquad time-split vs default path")
    # Where the two paths differ it is at the filter's own rounding-noise floor: a resonant low-cutoff biquad in
    # f32 direct form amplifies every rounding by ~1/(1 - r) ~ 10^3, and a start state that differs in the last
    # bit sends the recurrence down a different rounding trajectory.  Most voices agree far more closely.
    d = np.abs(plain[:, 3 * T:].astype(np.float64) - got[:, 3 * T:].astype(np.float64)).max(axis=1)
    assert float(np.median(d)) <= 2e-5


def test_time_split_mix_is_the_sum_of_the_rows():
    """With rows and a mix requested, a time-split block sums its output rows in voice order (two reduction
    kernels, fixed tree); against the oracle's sequential sum within the bus tolerance."""
    V, T = 300, 2048
    v = bank_for(0, V, 8 * T, mod_to_lpf_choices=(0.0,))
    v["active"][11::13] = 0
    ref, rbus, _ = oracle_bank_render(v, 0, [T, T])
    with s2.VoiceBank(v, SR, 0) as bank:
        bank.set_time_split(True)
        rows = torch.empty((V, T + 8), device="cuda", dtype=torch.float32)
        bus = torch.empty(2 * T, device="cuda", dtype=torch.float32)
        for i in range(2):
            bank.render(T, rows, T + 8, bus[i * T:(i + 1) * T])
        bank.sync()
        assert bank.time_split_blocks == 2
    got = bus.cpu().numpy()
    scale = max(1.0, float(np.max(np.abs(rbus))))
    assert float(np.max(np.abs(got - rbus))) <= TOL_ABS * scale
    assert_bus_within_bound(got[T:], rows[:, :T], V, "time_split", "second block")


def test_time_split_argument_errors():
    with s2.VoiceBank(bank_for(0, 64, 48000), SR, 0) as bank:
        bank.set_time_split(True)
        with pytest.raises(s2.S2Error):
            bank.set_pipeline(4)
        bank.set_time_split(False)
        bank.set_pipeline(2)
        with pytest.raises(s2.S2Error):
            bank.set_time_split(True)


# ------------------------------------------------------------------------------ patch files and scores

from synth2_b200 import patch as s2patch


def test_render_score_is_the_s2_bin_loop():
    """s2_synth_render_score == apply the events that arrived, then Synth::sample 16 frames (main.rs:138-147).
    Config-1 fixture plus events that arrive off the 16-frame grid; against the oracle's Synth driven chunk by
    chunk, and bit-for-bit against this library's own note_on / note_off / sample calls."""
    total = 60000
    raw = [(0, "on", 69), (1000, "on", 57), (12345, "on", 76), (24001, "off", 69), (40000, "off", 57), (40007, "off", 76),
           (59999, "on", 50)]                                   # the last one quantises to 60,000: never applied
    quantised = [((f + 15) & ~15, op, n) for f, op, n in raw]
    ref = run_script(oracle.OracleSynth(), total, quantised, chunk=16)
    syn = s2.Synth()
    got = syn.render_score(s2patch.make_events(raw), total, SR)
    assert_parity(ref, got, "render_score vs oracle Synth")
    stepwise = run_script(s2.Synth(), total, quantised)
    assert got.tobytes() == stepwise.tobytes()
    assert not syn.voice_info(3)[0]                             # note 50 was not started
    # the synth carries on: a second call continues the voices
    more = syn.render_score(s2patch.make_events([]), 4800, SR)
    assert more.shape == (4800,) and np.all(np.isfinite(more))
    syn.close()


@pytest.mark.parametrize("kind", ["one_pole", "biquad"])
def test_custom_patch_renders_like_the_oracle(kind):
    """A patch other than default_config(): every static_config::Layer field set, two overlapping notes.
    Expected = the oracle's process_layer_buf_simd per voice, mixed in slot order (synth.rs:176-202)."""
    text = f"""synth lead {{
        osc {{ kind square; gain 0.75 }}  noise 0.125
        lpf {{ freq 900; kind {kind}; damping 0.6 }}
        amp_env {{ attack 5; decay 40; sustain 0.625; release 120 }}
        mod_env {{ attack 2; decay 60; sustain 0.25; release 30 }}
        modulations {{ mod_env_to_lpf_freq 1.5 }}
    }}
    score {{ on 0 57; on 4800 64; off 14400 57; off 19200 64 }}"""
    p = s2patch.parse(text, SR)
    fk = p.filter_kind
    total = 28800
    syn = s2.Synth()
    syn.set_patch(p)
    got = syn.render_score(p.events, total, SR)
    syn.close()
    # oracle: one voice per note, each rendered from its own note-on
    mix = np.zeros(total, dtype=np.float32)
    for on, off, note in ((0, 14400, 57), (4800, 19200, 64)):
        v = np.zeros(1, dtype=s2.VOICE_DESC)
        v[0] = p.voice
        v["pitch_hz"] = s2.note_to_pitch(note)
        v["active"] = 1
        v["frame_offset"] = 0
        v["release_offset"] = off - on
        st = oracle.bank_init_states(v)
        o, _ = oracle.bank_render(v, st, SR, fk, total - on, want_bus=False)
        mix[on:] = mix[on:] + o[0]
    assert_parity(mix, got, f"custom patch ({kind})")
    assert np.max(np.abs(mix)) > 0.1


def test_set_patch_rules():
    syn = s2.Synth()
    bq = s2patch.parse("synth b { lpf { kind biquad; freq 500 } }")
    syn.note_on(60)
    with pytest.raises(s2.S2Error):
        syn.set_patch(bq)                                      # filter kind cannot change under a sounding voice
    syn.close()
    bad = s2patch.default_patch()
    bad.record["voice"]["amp_attack_ms"] = -1.0
    syn = s2.Synth()
    with pytest.raises(s2.S2Error):
        syn.set_patch(bad)
    with pytest.raises(s2.S2Error):
        syn.render_score(s2patch.make_events([(10, "on", 60), (5, "off", 60)]), 100, SR)
    syn.close()


def test_render_cli(tmp_path):
    from synth2_b200 import render
    src = tmp_path / "example.synth2"
    src.write_text("synth mySynth {\n\n}\n")
    out = tmp_path / "out.f32"
    assert render.main([str(src), "--seconds", "0.5", "--rate", "48000", "-o", str(out), "--note", "69"]) == 0
    got = np.fromfile(out, dtype="<f4")
    assert got.shape == (24000,)
    ref = run_script(oracle.OracleSynth(), 24000, [(0, "on", 69), (18000, "off", 69)])
    assert_parity(ref, got, "render CLI")
    wav = tmp_path / "out.wav"
    assert render.main([str(src), "--seconds", "0.1", "-o", str(wav)]) == 0
    assert wav.read_bytes()[:4] == b"RIFF"


def test_bench_times_the_steps_asked_and_dumps_the_last():
    """bench.py --steps K times K steps, and --dump-outputs writes what the last of them rendered: the same bank
    rendered here through the same pipelined path gives the same bits, and the oracle the same phases."""
    import json, pathlib, subprocess, sys, tempfile
    root = pathlib.Path(__file__).resolve().parent.parent
    V, T, K = 4096, 1024, 3
    with tempfile.TemporaryDirectory() as out:
        res = subprocess.run([sys.executable, str(root / "bench.py"), "--voices", str(V), "--block", str(T),
                              "--steps", str(K), "--warmup", "1", "--no-e2e", "--no-extra", "--no-cpu-baseline",
                              "--no-parity", "--dump-outputs", out], capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr
        rows, phase = np.load(pathlib.Path(out) / "last_block.npy"), np.load(pathlib.Path(out) / "phase.npy")
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and len(line["step_ms"]) == K and line["config"]["render_frames"] == K * T
    assert rows.dtype == np.float32 and rows.shape == (V, T) and phase.shape == (V,)
    v = bankgen.make_bank(V, 60 * SR, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    out = torch.empty((V, T), device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 1) as bank:
        bank.set_pipeline(4)
        for _ in range(K):
            bank.render(T, out, T, None)
        bank.sync()
    assert out.cpu().numpy().tobytes() == rows.tobytes()
    _, _, rst = oracle_bank_render(v, 1, [T] * K)
    assert rst["phase"].tobytes() == phase.tobytes()


# ------------------------------------------------------------------------------ player hand-off

def test_player_fill_is_the_reference_callback():
    """audio_player.rs `fill_buffer`: mono -> all channels, at most one new buffer per callback, zeros on
    underrun; the synth thread applies the notes that arrived before it renders a buffer (main.rs:138-147)."""
    B = s2.player.BUFFER_FRAMES
    with s2.Player(SR, start=False) as pl:
        out = np.full((512, 2), 7.0, np.float32)
        assert pl.fill(out) == 0 and np.all(out == 0.0)               # nothing rendered yet: zeros, counted
        assert pl.stats()["underruns"] == 1
        pl.note_on(69)
        pl.start()
        assert pl.wait_buffers(2)                                      # both buffers in circulation are filled
        ref = run_script(oracle.OracleSynth(), 3 * B, [(0, "on", 69)])
        got = []
        # callbacks of 600 stereo frames: buffer boundaries fall inside a callback
        for _ in range(8):
            out = np.full((600, 2), 7.0, np.float32)
            n = pl.fill(out)
            assert np.array_equal(out[:, 0], out[:, 1])
            assert np.all(out[n:] == 0.0)
            got.append(out[:n, 0].copy())
            pl.wait_buffers(pl.stats()["buffers_rendered"] + 1, 200)   # let the synth thread refill
        got = np.concatenate(got)
        assert got.size >= 2 * B
        assert_parity(ref[:got.size], got, "player stream")
        # a callback larger than a buffer takes one buffer and pads (audio_player.rs:150-152)
        pl.wait_buffers(pl.stats()["buffers_rendered"] + 2, 500)
        big = np.full(3 * B, 7.0, np.float32)
        n = pl.fill(big)
        assert n <= 2 * B and np.all(big[n:] == 0.0)
        st = pl.stats()
        assert st["frames_played"] == got.size + n and st["buffers_rendered"] >= 4


def test_player_note_off_and_patch():
    p = s2patch.parse("synth s { osc { kind sine } lpf { freq 4000 } amp_env { attack 1; decay 1; sustain 1; release 5 } "
                      "mod_env { decay 0 } modulations { mod_env_to_lpf_freq 0 } }")
    with s2.Player(SR, patch=p, start=False) as pl:
        pl.note_on(60)
        pl.start()
        assert pl.wait_buffers(2)
        pl.note_off(60)                                                # applied before the third buffer
        mono = np.zeros(s2.player.BUFFER_FRAMES, np.float32)
        chunks = []
        for _ in range(4):
            n = pl.fill(mono)
            chunks.append(mono[:n].copy())
            pl.wait_buffers(pl.stats()["buffers_rendered"] + 1, 300)
        x = np.concatenate(chunks)
        assert x.size == 4 * s2.player.BUFFER_FRAMES
        assert np.max(np.abs(x[:4096])) > 0.5                          # sounding
        assert np.all(x[3 * 2048 + 1024:] == 0.0)                      # released 5 ms into the third buffer
        with pytest.raises(s2.S2Error):
            lib_rc = s2.lib().s2_player_set_patch(pl._h, s2._lib.ptr(p.record))
            s2._lib.check(lib_rc)                                      # after start


# ------------------------------------------------------------------------------ out-of-bounds guards

@pytest.mark.parametrize("mode", ["default", "pipelined", "time_split"])
@pytest.mark.parametrize("V,frames", [(70, 1024), (1000, 2048), (33, 1000)])
def test_no_write_outside_the_output_rows(mode, V, frames):
    """Guard rows before / after the output block and guard columns after each row's `frames` must keep their
    sentinel: the transposed write-back, the ragged tail, the inactive-row clearing and the time-split
    segments all stay inside [row, row + frames)."""
    if mode == "time_split" and frames % 1024:
        pytest.skip("time-split needs whole 1,024-frame multiples (falls back otherwise: covered by 'default')")
    v = bank_for(0, V, 8 * frames, mod_to_lpf_choices=(0.0,))
    v["active"][3::7] = 0
    stride = ((frames + 3) & ~3) + 8
    buf = torch.full((V + 2, stride), -777.0, device="cuda", dtype=torch.float32)
    bus = torch.full((frames + 64,), -777.0, device="cuda", dtype=torch.float32)
    with s2.VoiceBank(v, SR, 0) as bank:
        if mode == "pipelined":
            bank.set_pipeline(3)
        if mode == "time_split":
            bank.set_time_split(True)
        for _ in range(2):
            bank.render(frames, buf[1:], stride, bus[32:])
        bank.sync()
        if mode == "time_split":
            assert bank.time_split_blocks == 2
    out = buf.cpu().numpy()
    assert np.all(out[0] == -777.0) and np.all(out[-1] == -777.0)
    assert np.all(out[1:-1, frames:] == -777.0)
    assert np.all(np.isfinite(out[1:-1, :frames])) and not np.any(out[1:-1, :frames] == -777.0)
    b = bus.cpu().numpy()
    assert np.all(b[:32] == -777.0) and np.all(b[32 + frames:] == -777.0)
    assert not np.any(b[32:32 + frames] == -777.0)


# ------------------------------------------------------------------------------ the rest of dsp_filters.rs

@pytest.mark.parametrize("filter_kind", [s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP, s2.FILTER_FIRST_ORDER_LP,
                                         s2.FILTER_FIRST_ORDER_HP])
def test_remaining_dsp_filters_against_oracle(filter_kind):
    """SecondOrderHighPass / SecondOrderBandPass / FirstOrderLowPass / FirstOrderHighPass (dsp_filters.rs:12-80,
    132-230) as the voice filter: sustain, moving cutoff, ramps, ragged blocks and the bus, against the oracle."""
    V = 96
    blocks = [4096, 4096, 2048, 1000, 3096]
    v = bankgen.make_bank(V, sum(blocks), kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE),
                          mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    v["noise_amt"][::3] = 0.25
    if filter_kind == s2.FILTER_BIQUAD_BP:
        v["damping"] += 2.0        # the field is the quality factor here; theta / (2 Q) must stay below pi / 4
    ref, rbus, rst = oracle_bank_render(v, filter_kind, blocks)
    assert np.all(np.isfinite(ref))
    got, gbus, st = gpu_bank_render(v, filter_kind, blocks)
    assert_parity(ref, got, f"filter kind {filter_kind}")
    assert st["phase"].tobytes() == rst["phase"].tobytes()
    for k in ("x1", "y1") + (("x2", "y2") if filter_kind in (s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP) else ()):
        np.testing.assert_allclose(st[k], rst[k], atol=TOL_ABS * 4, rtol=0)
    scale = max(1.0, float(np.max(np.abs(rbus))))
    assert float(np.max(np.abs(gbus - rbus))) <= TOL_ABS * scale
    # pipelined voice ranges give the same bits
    with s2.VoiceBank(v, SR, filter_kind) as bank:
        bank.set_pipeline(2)
        out = torch.empty((V, 4096), device="cuda", dtype=torch.float32)
        bank.render(4096, out, 4096, None)
        bank.sync()
        assert out.cpu().numpy().tobytes() == got[:, :4096].tobytes()
        with pytest.raises(s2.S2Error):
            bank.set_time_split(True)


def test_patch_selects_the_remaining_filters():
    p = s2patch.parse("synth hp { osc { kind saw } lpf { freq 700; kind biquad_hp; damping 0.9 } "
                      "mod_env { decay 0 } modulations { mod_env_to_lpf_freq 0 } } score { on 0 60; off 9600 60 }")
    assert p.filter_kind == s2.FILTER_BIQUAD_HP
    syn = s2.Synth()
    syn.set_patch(p)
    got = syn.render_score(p.events, 14400, SR)
    syn.close()
    vd = np.zeros(1, dtype=s2.VOICE_DESC)
    vd[0] = p.voice
    vd["pitch_hz"] = s2.note_to_pitch(60); vd["active"] = 1; vd["release_offset"] = 9600
    o, _ = oracle.bank_render(vd, oracle.bank_init_states(vd), SR, s2.FILTER_BIQUAD_HP, 14400, want_bus=False)
    assert_parity(o[0], got, "high-pass patch")


def test_compiled_example_renders_like_the_python_mirror(tmp_path):
    """examples/render_patch.cpp drives the C ABI from C++ (no Python in the process)."""
    import subprocess
    from test_host_logic import build_example
    exe = build_example(tmp_path)
    text = ("synth s { osc { kind triangle } lpf { freq 600 } } "
            "score { on 0 60; on 2400 64; off 9600 60; off 12000 64 }")
    (tmp_path / "p.synth2").write_text(text)
    res = subprocess.run([str(exe), str(tmp_path / "p.synth2"), "0.5", "48000", str(tmp_path / "o.f32")],
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    got = np.fromfile(tmp_path / "o.f32", dtype="<f4")
    p = s2patch.parse(text, SR)
    syn = s2.Synth()
    syn.set_patch(p)
    want = syn.render_score(p.events, 24000, SR)
    syn.close()
    assert got.tobytes() == want.tobytes()


def test_time_split_with_note_events_between_blocks():
    """release_voice / set_releases / set_voice between time-split blocks: the host's view of the voices (which
    decides whether a block qualifies and whether its cutoff moves) follows every edit."""
    V, T = 64, 2048
    v = bank_for(0, V, 16 * T)
    v["release_offset"] = s2.NO_RELEASE
    v["mod_sustain"] = 0.5
    v["mod_release_ms"] = 15.0
    ref_v = v.copy()
    st = oracle.bank_init_states(ref_v)
    outs_ref, outs = [], []
    with s2.VoiceBank(v, SR, 0) as bank:
        bank.set_time_split(True)

        def block():
            o, _ = oracle.bank_render(ref_v, st, SR, 0, T, want_bus=False)
            outs_ref.append(o)
            vo = torch.empty((V, T), device="cuda", dtype=torch.float32)
            bank.render(T, vo, T, None)
            bank.sync()
            outs.append(vo.cpu().numpy())

        for _ in range(6):                       # decay (moving cutoff), then sustain
            block()
        bank.release_voice(5)                    # note_off of one voice at frame 12,288
        ref_v["release_offset"][5] = 6 * T
        block()
        rel = np.full(V, s2.NO_RELEASE, dtype=np.uint32)
        rel[::2] = 7 * T + 100                   # bulk note-off table: half the voices, mid-block
        rel[5] = 6 * T
        bank.set_releases(rel)
        ref_v["release_offset"] = rel
        block(); block()
        nv = bank_for(0, 1, 16 * T)[0:1].copy()  # a new note in slot 9
        nv["pitch_hz"] = 523.25
        bank.set_voice(9, nv)
        ref_v[9] = nv[0]
        st[9] = oracle.bank_init_states(nv)[0]
        block(); block()
        assert bank.time_split_blocks == 11
        gst = bank.get_state()
    assert_parity(np.concatenate(outs_ref, axis=1), np.concatenate(outs, axis=1), "time-split with events")
    assert_state_parity(gst, st, 0)


@pytest.mark.timeout(120)
def test_player_lifecycle_stress():
    """Create / start / play / free many players in a row, with notes posted from another thread while the audio
    callback drains: no hang, no lost buffer, underruns only while nothing was rendered yet."""
    import threading
    for round_ in range(8):
        pl = s2.Player(SR, start=(round_ % 2 == 0))
        stop = threading.Event()

        def poster():
            k = 0
            while not stop.is_set():
                pl.note_on(40 + (k % 40))
                if k % 3 == 2:
                    pl.note_off(40 + ((k - 2) % 40))
                k += 1

        t = threading.Thread(target=poster)
        t.start()
        if round_ % 2:
            pl.start()
        out = np.zeros((512, 2), np.float32)
        got = 0
        for _ in range(24):
            got += pl.fill(out)
            assert np.all(np.isfinite(out))
        stop.set()
        t.join()
        st = pl.stats()
        assert st["frames_played"] == got
        assert st["buffers_rendered"] >= got // s2.player.BUFFER_FRAMES
        pl.close()
        pl.close()                                 # idempotent
