"""The oracle away from 48 kHz: every constant the render derives depends on the sample rate (period and phase step,
envelope stage boundaries of ms * sr / 1000, which are half-integers at 11.025 kHz, the cutoff's angle 2 pi f / sr),
so whole x16 blocks of the default patch are pinned against the independent numpy restatement of process.rs at
other rates, and at pitches the 48 kHz suite never reaches: at and above the sample rate (MIDI 120 and 127 at 8 kHz)
and around one and two times the rate."""
import numpy as np
import pytest

import oracle
from test_oracle_kats import _x16_block_numpy

L = oracle.lib()


def _f32(x):
    return float(np.float32(x))


def _ulp_below(x):
    return float(np.nextafter(np.float32(x), np.float32(0)))


def _ulp_above(x):
    return float(np.nextafter(np.float32(x), np.float32(np.inf)))


CASES = [(sr, 440.0) for sr in (8000, 11025, 12345, 22050, 44100, 96000, 192000)] + [
    (8000, _f32(L.s2o_note_to_pitch(120))),          # 8.37 kHz: above the rate
    (8000, _f32(L.s2o_note_to_pitch(127))),          # 12.5 kHz
    (8000, _f32(L.s2o_note_to_pitch(108))),          # 4.19 kHz: just above Nyquist
    (11025, _f32(L.s2o_note_to_pitch(125))),         # 11.2 kHz: above the rate
    (48000, _ulp_below(48000.0)), (48000, 48000.0), (48000, _ulp_above(48000.0)),
    (48000, _ulp_below(96000.0)), (48000, _ulp_above(96000.0)),
    (48000, 24000.0), (48000, _ulp_below(24000.0)),
]


def _config():
    cfg = oracle.default_config()
    c = cfg[0]
    assert c["osc_kind"] == 1 and c["filter_kind"] == 0 and c["mod_env_to_lpf_freq"] != 0.0
    env = lambda e: {"attack": e["attack_ms"], "decay": e["decay_ms"], "sustain": e["sustain"], "release": e["release_ms"]}
    cfg_n = {"osc_gain": c["osc_gain"], "noise": c["noise"], "lpf_freq": c["lpf_freq"],
             "mod_env_to_osc_freq": c["mod_env_to_osc_freq"], "mod_env_to_lpf_freq": c["mod_env_to_lpf_freq"],
             "amp_env": env(c["amp_env"]), "mod_env": env(c["mod_env"])}
    return cfg, cfg_n


@pytest.mark.parametrize("sr,pitch", CASES, ids=[f"{sr}-{p!r}" for sr, p in CASES])
def test_x16_blocks_at_other_rates_match_the_numpy_restatement(sr, pitch):
    """The default patch (saw, one-pole, 200 ms cutoff sweep of 10 octaves, amp 100/100/0.5/100 ms) from the note-on
    through the whole sweep, the sustain and a release that lands inside a block, to the end of the release: the
    oracle's s2o_process_layer_x16 against the numpy float32 restatement, bit for bit, output and carried phase."""
    cfg, cfg_n = _config()
    release = int(0.22 * sr) | 5                          # after the sweep, not on a block boundary
    end = release + int(0.1 * sr) + 64                    # past the end of the 100 ms release
    st_o = np.zeros(1, dtype=oracle.LAYER_STATE)
    st_n = {"phase": np.float32(0), "has_phase": 0, "lpf_last": np.float32(0), "noise_seed": 0}
    out_o = np.zeros(16, dtype=np.float32)
    for off in range(0, end, 16):
        L.s2o_process_layer_x16(cfg.ctypes.data, st_o.ctypes.data, pitch, sr, off, release, out_o.ctypes.data)
        with np.errstate(all="ignore"):                   # fmod / division at the edges of the phase step
            out_n = _x16_block_numpy(cfg_n, st_n, pitch, sr, off, release)
        assert out_o.tobytes() == out_n.tobytes(), f"block at offset {off}: {out_o} vs {out_n}"
        assert np.all(np.isfinite(out_o)), f"block at offset {off}"
        assert np.float32(st_o["phase"][0]).tobytes() == np.float32(st_n["phase"]).tobytes()
    assert np.all(out_o == 0.0)                           # silent after the release


def test_pitches_at_and_above_the_rate_exist_at_low_rates():
    """The cases above reach the pitch bands they are meant to: notes from 120 up are at or above 8 kHz, notes from
    108 up above its Nyquist frequency, notes from 125 up at or above 11.025 kHz."""
    pitch = [float(L.s2o_note_to_pitch(n)) for n in range(128)]
    assert min(n for n in range(128) if pitch[n] >= 8000.0) == 120
    assert min(n for n in range(128) if pitch[n] > 4000.0) == 108
    assert min(n for n in range(128) if pitch[n] >= 11025.0) == 125
