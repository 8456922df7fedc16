"""Kernel launches per API call, counted by s2_launch_count (bench.py reports them as launches_per_step).

The count is the shape of the host layer's stream graph: which kernels a call issues in each render mode (one stream,
pipelined voice ranges, time-split blocks), with and without output rows and bus, and when a note-off table staged
for a pipelined render is applied.  Expected counts:

    render, one stream      1, + 1 bus reduction when the bank is wider than one warp (32 voices)
    render, n_sub ranges    min(ceil(V / 64), n_sub), + 1 bus reduction above 32 voices (a copy at or below)
    time-split block        phase pre-pass + render, + 1 bus mix
    trace_phase             1, + 1 when a pipelined table is pending
    set_releases            0 when pipelined; else 0 in identity slot order (always at <= 32 voices), else 1 gather
    set_voice, release_voice, set_pipeline      1 when a pipelined table is pending, else 0
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import synth2_b200 as s2  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402

pytestmark = pytest.mark.gpu

SR = 48000
T = 1024                       # one time-split block
WIDTHS = (1, 32, 33, 2048, 65536)
MODES = (1, 2, 4, "ts")        # pipeline n_sub, or time-split on (one stream)
CASES = [(V, m) for V in WIDTHS for m in MODES if not (m == "ts" and V > 16384)]   # time-split: narrow banks only


def _launches(fn, *args):
    n0 = s2.lib().s2_launch_count()
    fn(*args)
    return s2.lib().s2_launch_count() - n0


def _render_launches(V, n_sub, split, bus):
    if split:
        return 2 + int(bus)
    return min(-(-V // 64), n_sub) + int(bus and V > 32)


def _open(V, mode):
    bank = s2.VoiceBank(bankgen.make_bank(V, 1 << 20), SR, s2.FILTER_ONE_POLE)
    if mode == "ts":
        bank.set_time_split(True)
        return bank, 1
    bank.set_pipeline(mode)
    return bank, mode


@pytest.mark.parametrize("V,mode", CASES)
def test_render_launches(V, mode):
    rows = torch.empty((V, T), device="cuda:0", dtype=torch.float32)
    bus = torch.empty(T, device="cuda:0", dtype=torch.float32)
    host = np.empty(T, np.float32)
    pinned = torch.empty(T, dtype=torch.float32).pin_memory()
    bank, n_sub = _open(V, mode)
    with bank:
        for frames in (T, 1000):                       # 1,000 frames is no time-split block
            for want_rows in (False, True):
                for want_bus in (False, True):
                    split = mode == "ts" and want_rows and frames % 1024 == 0
                    b0 = bank.time_split_blocks
                    got = _launches(bank.render, frames, rows if want_rows else None, T, bus if want_bus else None)
                    assert got == _render_launches(V, n_sub, split, want_bus), (frames, want_rows, want_bus)
                    assert bank.time_split_blocks - b0 == int(split)
            for want_rows in (False, True):
                split = mode == "ts" and want_rows and frames % 1024 == 0
                r = rows if want_rows else None
                assert _launches(bank.render_bus_host, frames, r, T, host) == _render_launches(V, n_sub, split, True)
                assert _launches(bank.render_bus_host_async, frames, pinned, r, T) == \
                    _render_launches(V, n_sub, split, True)
            assert _launches(bank.trace_phase, frames, rows, T) == 1
        bank.sync()


@pytest.mark.parametrize("V,mode", CASES)
def test_staged_table_launches(V, mode):
    """A table set between renders, then each entry that settles it: the pipelined render applies it in its own
    launches, the other entries with one gather first.  Either way it is applied once."""
    rows = torch.empty((V, T), device="cuda:0", dtype=torch.float32)
    bus = torch.empty(T, device="cuda:0", dtype=torch.float32)
    table = np.full(V, 3 * T, np.uint32)
    voices = bankgen.make_bank(V, 1 << 20)
    bank, n_sub = _open(V, mode)
    pending = n_sub > 1
    staged = 0 if pending else int(V > 32)             # make_bank's mixed kinds permute the slots above 32 voices
    settlers = {
        "set_voice": (lambda: bank.set_voice(V - 1, voices[V - 1:]), 0),
        "release_voice": (lambda: bank.release_voice(0), 0),
        "trace_phase": (lambda: bank.trace_phase(T, rows, T), 1),
        "set_pipeline": (lambda: bank.set_pipeline(n_sub), 0),
        "render": (lambda: bank.render(T, rows, T, bus), _render_launches(V, n_sub, mode == "ts", True)),
    }
    with bank:
        for name, (entry, alone) in settlers.items():
            assert _launches(bank.set_releases, table) == staged
            if pending:                                # a second table before any render supersedes the first
                assert _launches(bank.set_releases, table) == 0
            extra = int(pending and name != "render")
            assert _launches(entry) == alone + extra, name
            assert _launches(bank.release_voice, 1 % V) == 0, name   # nothing is left pending
        bank.sync()


def test_set_releases_identity_order():
    """Above 32 voices the gather runs only when the slot order differs from the voice order."""
    same = bankgen.make_bank(33, 1 << 20, kinds=(s2.OSC_SAW,), mod_to_lpf_choices=(0.0,))
    same["amp_attack_ms"] = 10.0
    same["amp_decay_ms"] = 10.0
    mixed = bankgen.make_bank(33, 1 << 20)
    table = np.full(33, 3 * T, np.uint32)
    for voices, expect in ((same, 0), (mixed, 1)):
        with s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE) as bank:
            assert _launches(bank.set_releases, table) == expect
            bank.sync()
