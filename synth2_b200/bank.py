"""VoiceBank — host-side handle of s2_bank: V independent voices resident on one GPU.

Mirrors `process::process_layer_buf_simd(&sc::Layer, &mut st::Layer, pitch, sample_rate, offset,
release_offset, buf)` (s2_lib/src/try3/process.rs:14-22) batched over voices: each render call
fills `frames` frames per voice (x16 blocks then the `frames % 16` scalar tail) and carries
`st::Layer` + the frame offset to the next call.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import VOICE_DESC, VOICE_STATE, check, lib, ptr


def note_to_pitch(note: int) -> float:
    """synth.rs:208-212 (host libm powf inside libs2cuda.so)."""
    return float(lib().s2_note_to_pitch(int(note) & 0xFF))


def _row_stride(buf, frames: int, given: int) -> int:
    """The row stride in floats: `given` if set, else the buffer's own (a tensor's stride(0)), else `frames`."""
    if given or buf is None:
        return int(given)
    return int(buf.stride(0)) if hasattr(buf, "stride") else int(frames)


def _stream_ptr(stream):
    """A torch stream, a raw cudaStream_t or None (the default stream) as the library's `void* stream`."""
    return None if stream is None else C.c_void_p(getattr(stream, "cuda_stream", stream))


def default_voice(n: int = 1) -> np.ndarray:
    """`Synth::default_config()` (synth.rs:125-152) as n inactive voice descriptions."""
    one = np.zeros(1, dtype=VOICE_DESC)
    lib().s2_default_voice(ptr(one))
    return np.repeat(one, n)


class VoiceBank:
    def __init__(self, voices: np.ndarray, sample_rate: int = 48000,
                 filter_kind: int = _lib.FILTER_ONE_POLE, device: int = 0, stream=None):
        voices = self._setup(voices, sample_rate, filter_kind, device)
        check(lib().s2_bank_create(self.device, self.sample_rate, self.filter_kind, self.n_voices,
                                   ptr(voices), _stream_ptr(stream), C.byref(self._h)))

    def _setup(self, voices, sample_rate, filter_kind, device) -> np.ndarray:
        """The handle and fields every bank has, before s2_bank_create(_mixed) fills the handle; returns the voices
        as the contiguous array the library reads."""
        voices = np.ascontiguousarray(voices, dtype=VOICE_DESC)
        self._h = C.c_void_p()
        self.n_voices = int(voices.shape[0])
        self.sample_rate = int(sample_rate)
        self.filter_kind = int(filter_kind)
        self.device = int(device)
        return voices

    @classmethod
    def mixed(cls, voices: np.ndarray, filter_kinds, sample_rate: int = 48000, device: int = 0, stream=None):
        """A bank whose voice i renders through filter filter_kinds[i] (s2_bank_create_mixed).  `filter_kind` is then
        the kind of voice 0; `filter_kinds` has them all."""
        voices = np.asarray(voices).reshape(-1)
        kinds = np.asarray(filter_kinds).reshape(-1)
        if kinds.size != voices.size:
            raise ValueError(f"{kinds.size} filter kinds for {voices.size} voices")
        if kinds.size and (kinds.min() < 0 or kinds.max() > 0xFFFFFFFF):
            raise ValueError("filter kind out of range")
        kinds = np.ascontiguousarray(kinds, dtype=np.uint32)
        self = cls.__new__(cls)
        voices = self._setup(voices, sample_rate, kinds[0] if kinds.size else 0, device)
        check(lib().s2_bank_create_mixed(self.device, self.sample_rate, self.n_voices, ptr(voices), ptr(kinds),
                                         _stream_ptr(stream), C.byref(self._h)))
        return self

    @classmethod
    def routed(cls, voices: np.ndarray, filter_kinds, bus_of_voice, n_buses: int = None, sample_rate: int = 48000,
               device: int = 0, stream=None):
        """A bank whose voice i renders through filter filter_kinds[i] and mixes into bus bus_of_voice[i]
        (s2_bank_create_routed); n_buses defaults to max(bus_of_voice) + 1.  render(..., buses=...) writes every bus."""
        voices = np.asarray(voices).reshape(-1)
        kinds = np.asarray(filter_kinds).reshape(-1)
        buses = np.asarray(bus_of_voice).reshape(-1)
        if kinds.size != voices.size or buses.size != voices.size:
            raise ValueError(f"{kinds.size} filter kinds and {buses.size} buses for {voices.size} voices")
        if kinds.size and (kinds.min() < 0 or kinds.max() > 0xFFFFFFFF):
            raise ValueError("filter kind out of range")
        if buses.size and (buses.min() < 0 or buses.max() > 0xFFFFFFFF):
            raise ValueError("bus out of range")
        if n_buses is None:
            n_buses = int(buses.max()) + 1 if buses.size else 1
        if not 0 <= int(n_buses) <= 0xFFFFFFFF:
            raise ValueError("n_buses out of range")
        kinds = np.ascontiguousarray(kinds, dtype=np.uint32)
        buses = np.ascontiguousarray(buses, dtype=np.uint32)
        self = cls.__new__(cls)
        voices = self._setup(voices, sample_rate, kinds[0] if kinds.size else 0, device)
        check(lib().s2_bank_create_routed(self.device, self.sample_rate, self.n_voices, ptr(voices), ptr(kinds),
                                          ptr(buses), int(n_buses), _stream_ptr(stream), C.byref(self._h)))
        return self

    @property
    def n_buses(self) -> int:
        """Buses of the bank: 1 unless it is routed."""
        n = C.c_uint32(0)
        check(lib().s2_bank_buses(self._h, C.byref(n), None))
        return int(n.value)

    @property
    def bus_of_voice(self) -> np.ndarray:
        """The bus of every voice, in voice order (np.uint32)."""
        out = np.zeros(self.n_voices, dtype=np.uint32)
        check(lib().s2_bank_buses(self._h, None, ptr(out)))
        return out

    @property
    def filter_kinds(self) -> np.ndarray:
        """The filter kind of every voice, in voice order (np.uint32)."""
        out = np.zeros(self.n_voices, dtype=np.uint32)
        check(lib().s2_bank_filter_kinds(self._h, ptr(out)))
        return out

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().s2_bank_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- voices
    def set_voice(self, index: int, voice: np.ndarray):
        voice = np.ascontiguousarray(voice, dtype=VOICE_DESC).reshape(-1)[:1]
        check(lib().s2_bank_set_voice(self._h, int(index), ptr(voice)))

    def set_voices(self, indices, voices: np.ndarray):
        """Bulk note_on: the same as set_voice(indices[j], voices[j]) for j = 0, 1, ... in order (the last entry of a
        repeated index wins), applied on the GPU without waiting for the bank's renders."""
        idx = np.asarray(indices).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() > 0xFFFFFFFF):
            raise IndexError("voice index out of range")
        idx = np.ascontiguousarray(idx, dtype=np.uint32)
        voices = np.ascontiguousarray(voices, dtype=VOICE_DESC).reshape(-1)
        if voices.size != idx.size:
            raise ValueError(f"{idx.size} indices for {voices.size} voices")
        check(lib().s2_bank_set_voices(self._h, idx.size, ptr(idx), ptr(voices)))

    def release_voice(self, index: int):
        check(lib().s2_bank_release_voice(self._h, int(index)))

    def set_releases(self, release_offsets):
        """Bulk note_off table: u32 per voice (NO_RELEASE = held); numpy array or pinned torch tensor."""
        check(lib().s2_bank_set_releases(self._h, ptr(release_offsets)))

    # -- rendering (device buffers: anything with .data_ptr(), or a raw address)
    def render(self, frames: int, voice_out=None, row_stride: int = 0, bus_out=None, sum_sq=None, peak=None,
               buses=None, bus_stride: int = 0):
        """Render `frames` frames.  With `sum_sq` and `peak` (per-voice meters, given together: float64 and float32 device
        tensors of n_voices, or raw addresses) every active voice also adds its sum of y*y to sum_sq and raises peak to
        its largest |y| (s2_bank_render_metered); voice_out and bus_out may then both be None.  With `buses` (a device
        tensor of n_buses rows, or a raw address) bus g goes to row g, `bus_stride` floats apart (default: the tensor's
        stride(0)), instead of one bus_out (s2_bank_render_buses)."""
        row_stride = _row_stride(voice_out, frames, row_stride)
        if sum_sq is None and peak is None and buses is None:
            check(lib().s2_bank_render(self._h, int(frames), ptr(voice_out), row_stride, ptr(bus_out)))
            return
        if (sum_sq is None) != (peak is None):
            raise ValueError("sum_sq and peak are given together")
        for m, dtype in ((sum_sq, "float64"), (peak, "float32")):
            if hasattr(m, "data_ptr") and (str(m.dtype) != "torch." + dtype or m.numel() != self.n_voices
                                           or not m.is_contiguous()):
                raise ValueError(f"a meter is a contiguous {dtype} tensor of {self.n_voices} entries")
        if buses is not None:
            if bus_out is not None:
                raise ValueError("bus_out and buses are exclusive")
            if hasattr(buses, "data_ptr") and (str(buses.dtype) != "torch.float32" or buses.dim() != 2
                                               or buses.shape[0] != self.n_buses or buses.shape[1] < frames
                                               or buses.stride(1) != 1):
                raise ValueError(f"buses is a float32 tensor of {self.n_buses} rows of at least {frames} frames")
            check(lib().s2_bank_render_buses(self._h, int(frames), ptr(voice_out), row_stride, ptr(buses),
                                             _row_stride(buses, frames, bus_stride), ptr(sum_sq), ptr(peak)))
            return
        check(lib().s2_bank_render_metered(self._h, int(frames), ptr(voice_out), row_stride, ptr(bus_out),
                                           ptr(sum_sq), ptr(peak)))

    def render_bus_host(self, frames: int, voice_out=None, row_stride: int = 0, out: np.ndarray = None):
        """Render and return the mono mix in host memory (the `Synth::sample` shape)."""
        if out is None:
            out = np.empty(int(frames), dtype=np.float32)
        assert out.dtype == np.float32 and out.flags.c_contiguous and out.size >= frames
        row_stride = _row_stride(voice_out, frames, row_stride)
        check(lib().s2_bank_render_bus_host(self._h, int(frames), ptr(voice_out), row_stride, ptr(out)))
        return out

    def render_bus_host_async(self, frames: int, pinned_out, voice_out=None, row_stride: int = 0):
        """Streaming form: enqueue render + mix + D2H of the mix into pinned host memory, no sync."""
        row_stride = _row_stride(voice_out, frames, row_stride)
        check(lib().s2_bank_render_bus_host_async(self._h, int(frames), ptr(voice_out), row_stride, ptr(pinned_out)))

    def trace_phase(self, frames: int, phase_out, row_stride: int = 0):
        check(lib().s2_bank_trace_phase(self._h, int(frames), ptr(phase_out), _row_stride(phase_out, frames, row_stride)))

    def sync(self):
        check(lib().s2_bank_sync(self._h))

    def set_pipeline(self, n_sub: int):
        """n_sub > 1: render contiguous voice ranges on n_sub internal streams (see include/s2_cuda.h)."""
        check(lib().s2_bank_set_pipeline(self._h, int(n_sub)))

    def set_time_split(self, enable: bool = True):
        """Narrow banks: render qualifying blocks as 32 time segments per voice (s2_cuda.h)."""
        check(lib().s2_bank_set_time_split(self._h, 1 if enable else 0))

    @property
    def time_split_blocks(self) -> int:
        """Blocks rendered through the time-split kernels so far."""
        n = C.c_uint64(0)
        check(lib().s2_bank_time_split_blocks(self._h, C.byref(n)))
        return int(n.value)

    def join(self, stream=None):
        """Make `stream` (a torch stream, a raw cudaStream_t, or None = default) wait for the bank's work."""
        check(lib().s2_bank_join(self._h, _stream_ptr(stream)))

    # -- carried state
    def get_state(self) -> np.ndarray:
        st = np.zeros(self.n_voices, dtype=VOICE_STATE)
        check(lib().s2_bank_get_state(self._h, ptr(st)))
        return st

    def set_state(self, state: np.ndarray):
        state = np.ascontiguousarray(state, dtype=VOICE_STATE)
        assert state.shape[0] == self.n_voices
        check(lib().s2_bank_set_state(self._h, ptr(state)))
