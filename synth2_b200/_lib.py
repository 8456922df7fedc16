"""ctypes binding of libs2cuda.so — the C ABI in include/s2_cuda.h, nothing more.

There is no fallback: if the library is missing this module raises at import of the symbol
table, and every compute entry fails with an error from the library when no GPU is present.
"""
import ctypes as C
import pathlib

import numpy as np

PKG = pathlib.Path(__file__).resolve().parent
import os

LIB_PATH = pathlib.Path(os.environ["S2_LIB"]) if os.environ.get("S2_LIB") else PKG / "libs2cuda.so"   # S2_LIB: experiments only

S2_OK = 0
S2_ERR_INVALID = -1
S2_ERR_NO_DEVICE = -2
S2_ERR_CUDA = -3
S2_ERR_OVERFLOW = -4
S2_ERR_NOMEM = -5

OSC_SQUARE, OSC_SAW, OSC_TRIANGLE, OSC_SINE = 0, 1, 2, 3
FILTER_ONE_POLE, FILTER_BIQUAD_LP = 0, 1
FILTER_BIQUAD_HP, FILTER_BIQUAD_BP, FILTER_FIRST_ORDER_LP, FILTER_FIRST_ORDER_HP = 2, 3, 4, 5
NO_RELEASE = 0xFFFFFFFF
MAX_BUSES = 65536

# struct s2_voice_desc (80 bytes) / s2_voice_state (32 bytes), include/s2_cuda.h
VOICE_DESC = np.dtype([
    ("osc_kind", "<u4"), ("noise_seed", "<u4"), ("pitch_hz", "<f4"), ("osc_gain", "<f4"),
    ("noise_amt", "<f4"), ("lpf_freq_hz", "<f4"), ("damping", "<f4"),
    ("amp_attack_ms", "<f4"), ("amp_decay_ms", "<f4"), ("amp_sustain", "<f4"), ("amp_release_ms", "<f4"),
    ("mod_attack_ms", "<f4"), ("mod_decay_ms", "<f4"), ("mod_sustain", "<f4"), ("mod_release_ms", "<f4"),
    ("mod_env_to_osc_freq", "<f4"), ("mod_env_to_lpf_freq", "<f4"),
    ("frame_offset", "<u4"), ("release_offset", "<u4"), ("active", "<u4"),
])
VOICE_STATE = np.dtype([
    ("phase", "<f4"), ("has_phase", "<u4"), ("frame_offset", "<u4"), ("lpf_last", "<f4"),
    ("x1", "<f4"), ("x2", "<f4"), ("y1", "<f4"), ("y2", "<f4"),
])
# struct s2_patch (144 bytes) / s2_note_event (16 bytes)
PATCH = np.dtype([("voice", VOICE_DESC), ("filter_kind", "<u4"), ("name", "S60")])
NOTE_EVENT = np.dtype([("frame", "<u8"), ("note", "u1"), ("on", "u1"), ("reserved", "u1", (2,)), ("velocity", "<f4")])
assert VOICE_DESC.itemsize == 80 and VOICE_STATE.itemsize == 32
assert PATCH.itemsize == 144 and NOTE_EVENT.itemsize == 16

# every symbol include/s2_cuda.h declares: (restype, argtypes)
_vp, _sz, _u32, _u8, _f, _i = C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint8, C.c_float, C.c_int
SYMBOLS = {
    "s2_abi_version": (_u32, []),
    "s2_last_error": (C.c_char_p, []),
    "s2_device_count": (_i, [C.POINTER(_i)]),
    "s2_note_to_pitch": (_f, [_u8]),
    "s2_default_voice": (None, [_vp]),
    "s2_bank_create": (_i, [_i, _u32, _u32, _sz, _vp, _vp, C.POINTER(_vp)]),
    "s2_bank_create_mixed": (_i, [_i, _u32, _sz, _vp, _vp, _vp, C.POINTER(_vp)]),
    "s2_bank_create_routed": (_i, [_i, _u32, _sz, _vp, _vp, _vp, _u32, _vp, C.POINTER(_vp)]),
    "s2_bank_destroy": (None, [_vp]),
    "s2_bank_voices": (_sz, [_vp]),
    "s2_bank_filter_kinds": (_i, [_vp, _vp]),
    "s2_bank_buses": (_i, [_vp, C.POINTER(_u32), _vp]),
    "s2_bank_set_voice": (_i, [_vp, _sz, _vp]),
    "s2_bank_set_voices": (_i, [_vp, _sz, _vp, _vp]),
    "s2_bank_release_voice": (_i, [_vp, _sz]),
    "s2_bank_set_releases": (_i, [_vp, _vp]),
    "s2_bank_render": (_i, [_vp, _sz, _vp, _sz, _vp]),
    "s2_bank_render_metered": (_i, [_vp, _sz, _vp, _sz, _vp, _vp, _vp]),
    "s2_bank_render_buses": (_i, [_vp, _sz, _vp, _sz, _vp, _sz, _vp, _vp]),
    "s2_bank_render_bus_host": (_i, [_vp, _sz, _vp, _sz, _vp]),
    "s2_bank_render_bus_host_async": (_i, [_vp, _sz, _vp, _sz, _vp]),
    "s2_bank_get_state": (_i, [_vp, _vp]),
    "s2_bank_set_state": (_i, [_vp, _vp]),
    "s2_bank_sync": (_i, [_vp]),
    "s2_bank_set_pipeline": (_i, [_vp, _i]),
    "s2_bank_join": (_i, [_vp, _vp]),
    "s2_bank_set_time_split": (_i, [_vp, _i]),
    "s2_bank_time_split_blocks": (_i, [_vp, C.POINTER(C.c_uint64)]),
    "s2_bank_trace_phase": (_i, [_vp, _sz, _vp, _sz]),
    "s2_comm_version": (_i, [C.POINTER(_i)]),
    "s2_comm_unique_id": (_i, [_vp]),
    "s2_comm_create": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "s2_comm_adopt": (_i, [_vp, _i, _i, _i, C.POINTER(_vp)]),
    "s2_comm_destroy": (None, [_vp]),
    "s2_bank_reduce_bus": (_i, [_vp, _vp, _i, _vp, _vp, _sz, _vp]),
    "s2_launch_count": (C.c_uint64, []),
    "s2_synth_new": (_i, [_i, C.POINTER(_vp)]),
    "s2_synth_free": (None, [_vp]),
    "s2_synth_note_on": (_i, [_vp, _u8, _f]),
    "s2_synth_note_off": (_i, [_vp, _u8]),
    "s2_synth_sample": (_i, [_vp, _vp, _sz, _u32]),
    "s2_synth_voice_info": (_i, [_vp, _i, C.POINTER(_u8), C.POINTER(_u32), C.POINTER(_u32), _vp]),
    "s2_default_patch": (None, [_vp]),
    "s2_patch_parse": (_i, [C.c_char_p, _u32, _vp, _vp, _sz, C.POINTER(_sz)]),
    "s2_synth_set_patch": (_i, [_vp, _vp]),
    "s2_synth_render_score": (_i, [_vp, _vp, _sz, _u32, _vp, _sz]),
    "s2_player_new": (_i, [_i, _u32, C.POINTER(_vp)]),
    "s2_player_free": (None, [_vp]),
    "s2_player_set_patch": (_i, [_vp, _vp]),
    "s2_player_start": (_i, [_vp]),
    "s2_player_note_on": (_i, [_vp, _u8, _f]),
    "s2_player_note_off": (_i, [_vp, _u8]),
    "s2_player_fill": (C.c_int64, [_vp, _vp, _sz, _u32]),
    "s2_player_stats": (_i, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "s2_player_wait_buffers": (_i, [_vp, C.c_uint64, _u32]),
}


class S2Error(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libs2cuda error {code}: {message}")
        self.code = code


_lib = None


def lib():
    """Loads libs2cuda.so once.  Raises if it has not been built (python -m synth2_b200.build)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing: build it with `python -m synth2_b200.build` "
                              "(the renderer has no CPU or PyTorch fallback)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc < 0:
        raise S2Error(rc, lib().s2_last_error().decode("utf-8", "replace"))
    return rc


def ptr(a):
    """Address of a numpy array / torch tensor / int / None as a c_void_p."""
    if a is None:
        return None
    if isinstance(a, int):
        return C.c_void_p(a)
    if isinstance(a, np.ndarray):
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))
