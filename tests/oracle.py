"""ctypes binding of oracle/libs2oracle.so (the CPU restatement).  TEST INFRASTRUCTURE: imported by
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs only."""
import ctypes as C
import pathlib
import subprocess
import tempfile

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
SO = ROOT / "oracle" / "libs2oracle.so"

ADSR = np.dtype([("attack_ms", "<f4"), ("decay_ms", "<f4"), ("sustain", "<f4"), ("release_ms", "<f4")])
LAYER_CONFIG = np.dtype([
    ("osc_kind", "<u4"), ("osc_gain", "<f4"), ("noise", "<f4"), ("lpf_freq", "<f4"),
    ("amp_env", ADSR), ("mod_env", ADSR),
    ("mod_env_to_osc_freq", "<f4"), ("mod_env_to_lpf_freq", "<f4"),
    ("filter_kind", "<u4"), ("damping", "<f4"),
])
LAYER_STATE = np.dtype([("has_phase", "<u4"), ("phase", "<f4"), ("noise_seed", "<u4"), ("lpf_last", "<f4"),
                        ("x1", "<f4"), ("x2", "<f4"), ("y1", "<f4"), ("y2", "<f4")])
NO_RELEASE = 0xFFFFFFFF

_vp, _sz, _u32, _u8, _f, _i = C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint8, C.c_float, C.c_int
_SIGS = {
    "s2o_ms_as_samples": (_f, [_f, _u32]),
    "s2o_hz_as_samples": (_f, [_f, _u32]),
    "s2o_note_to_pitch": (_f, [_u8]),
    "s2o_hash_word": (_u32, [_u32, _u32]),
    "s2o_hash_word_x16": (None, [_vp, _vp, _vp]),
    "s2o_hash_noise": (_f, [_u32, _f]),
    "s2o_noise_fast_form": (_f, [_u32, _u32]),
    "s2o_line_fma": (_f, [_f, _f, _f, _f]),
    "s2o_line_nofma": (_f, [_f, _f, _f, _f]),
    "s2o_adsr_x16_lane": (_f, [_f, _f, _f, _f, _u32, _u32]),
    "s2o_adsr_scalar": (_f, [_f, _f, _f, _f, _u32, _u32]),
    "s2o_modulate_freq": (_f, [_f, _f, _f]),
    "s2o_accum_phase": (_f, [_f, _f]),
    "s2o_table_lookup_exclusive": (_f, [_vp, _u32, _f, _f, _i]),
    "s2o_table_lookup_inclusive": (_f, [_vp, _u32, _f, _f, _i]),
    "s2o_table_lookup_periodic": (_f, [_vp, _u32, _f, _f, _i]),
    "s2o_osc_sample": (_f, [_u32, _f, _f, _i]),
    "s2o_lpf_coeff": (_f, [_f, _u32]),
    "s2o_lpf_process": (_f, [_vp, _u32, _f, _f]),
    "s2o_biquad_lp_coeffs": (None, [_u32, _f, _f, _vp]),
    "s2o_biquad_lp_process": (_f, [_vp, _u32, _f, _f, _f]),
    "s2o_biquad_hp_process": (_f, [_vp, _u32, _f, _f, _f]),
    "s2o_biquad_bp_process": (_f, [_vp, _u32, _f, _f, _f]),
    "s2o_first_order_process": (_f, [_vp, _u32, _f, _i, _f]),
    "s2o_sin_table": (_vp, []),
    "s2o_process_layer_x16": (None, [_vp, _vp, _f, _u32, _u32, _u32, _vp]),
    "s2o_process_layer": (_f, [_vp, _vp, _f, _u32, _u32, _u32]),
    "s2o_process_layer_buf_simd": (_i, [_vp, _vp, _f, _u32, _u32, _u32, _vp, _sz]),
    "s2o_trace_voice": (None, [_vp, _f, _u32, _u32, _u32, _sz, _vp, _vp, _vp, _vp]),
    "s2o_synth_new": (_vp, []),
    "s2o_synth_free": (None, [_vp]),
    "s2o_synth_note_on": (None, [_vp, _u8, _f]),
    "s2o_synth_note_off": (_i, [_vp, _u8]),
    "s2o_synth_sample": (None, [_vp, _vp, _sz, _u32]),
    "s2o_synth_voice_info": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "s2o_default_config": (None, [_vp]),
    "s2o_bank_render": (_i, [_vp, _vp, _sz, _u32, _u32, _sz, _vp, _sz, _vp, _i]),
    "s2o_bank_init_states": (None, [_vp, _vp, _sz]),
}

_lib = None


def use_native_build():
    """bench.py only: time the CPU baseline on a build tuned for THIS host (`make -C oracle native`: -O3
    -march=native, same IEEE semantics).  Built fresh in a temporary directory, since the tree may be read-only
    and a copy built on another host may use other instructions.  Falls back to the portable library when it
    cannot be built.  Returns the flags description for the bench line."""
    global _lib
    try:
        with tempfile.TemporaryDirectory() as tmp:
            native = pathlib.Path(tmp) / "libs2oracle_native.so"
            subprocess.run(["make", "-C", str(ROOT / "oracle"), "native", f"NATIVE_SO={native}"],
                           check=True, capture_output=True)
            _lib = _load(native)                # stays mapped after the directory is removed
        return "-O3 -march=native -ffp-contract=off"
    except Exception:
        return "-O2 -march=x86-64-v3 -ffp-contract=off"


def _load(path):
    h = C.CDLL(str(path))
    for name, (res, args) in _SIGS.items():
        fn = getattr(h, name)
        fn.restype, fn.argtypes = res, args
    return h


def lib():
    global _lib
    if _lib is None:
        if not SO.exists():
            subprocess.run(["make", "-C", str(SO.parent)], check=True, capture_output=True)
        _lib = _load(SO)
    return _lib


def _p(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def sin_table():
    addr = lib().s2o_sin_table()
    return np.ctypeslib.as_array((C.c_float * 1024).from_address(addr)).copy()


def pitch_table():
    """128-entry f32 table of the oracle's `note_to_pitch` (synth.rs:208-212)."""
    return np.array([lib().s2o_note_to_pitch(n) for n in range(128)], dtype=np.float32)


def default_config():
    cfg = np.zeros(1, dtype=LAYER_CONFIG)
    lib().s2o_default_config(_p(cfg))
    return cfg


def bank_init_states(voices):
    from synth2_b200 import VOICE_STATE
    st = np.zeros(voices.shape[0], dtype=VOICE_STATE)
    lib().s2o_bank_init_states(_p(voices), _p(st), voices.shape[0])
    return st


def bank_render(voices, states, sample_rate, filter_kind, frames, want_voices=True, want_bus=True, nthreads=1):
    """Returns (voice_out [V, frames] or None, bus [frames] or None); advances `states` in place."""
    V = voices.shape[0]
    out = np.zeros((V, frames), dtype=np.float32) if want_voices else None
    bus = np.zeros(frames, dtype=np.float32) if want_bus else None
    rc = lib().s2o_bank_render(_p(voices), _p(states), V, sample_rate, filter_kind, frames,
                               _p(out), frames, _p(bus), nthreads)
    assert rc == 0, "oracle: frame offset overflow"
    return out, bus


def trace_voice(cfg, pitch, sample_rate, offset, release_offset, frames):
    """x16 render of one voice with debug taps: (out, phases, table_idx, final_state)."""
    assert frames % 16 == 0
    st = np.zeros(1, dtype=LAYER_STATE)
    out = np.zeros(frames, dtype=np.float32)
    ph = np.zeros(frames, dtype=np.float32)
    idx = np.zeros(frames, dtype=np.uint32)
    lib().s2o_trace_voice(_p(cfg), pitch, sample_rate, offset, release_offset, frames, _p(st), _p(ph), _p(idx), _p(out))
    return out, ph, idx, st


class OracleSynth:
    """synth::Synth restated on the CPU (oracle/s2_oracle.c)."""

    def __init__(self):
        self._h = C.c_void_p(lib().s2o_synth_new())

    def __del__(self):
        if self._h:
            lib().s2o_synth_free(self._h)
            self._h = None

    def note_on(self, note, velocity=1.0):
        lib().s2o_synth_note_on(self._h, note, velocity)

    def note_off(self, note):
        return lib().s2o_synth_note_off(self._h, note) == 1

    def sample(self, buffer, sample_rate):
        assert buffer.dtype == np.float32 and buffer.flags.c_contiguous
        lib().s2o_synth_sample(self._h, _p(buffer), buffer.size, sample_rate)

    def voice_info(self, slot):
        note, cur, rel = C.c_uint8(), C.c_uint32(), C.c_uint32()
        st = np.zeros(1, dtype=LAYER_STATE)
        used = lib().s2o_synth_voice_info(self._h, slot, C.byref(note), C.byref(cur), C.byref(rel), _p(st))
        return (bool(used), note.value, cur.value if used else None,
                None if rel.value == NO_RELEASE else rel.value, st[0])
