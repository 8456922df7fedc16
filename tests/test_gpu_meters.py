"""Per-voice level meters, s2_bank_render_metered: sum of squares and peak magnitude accumulated in the render kernel.

    rows            the meters of a call against the rows that call rendered: peak bits exact, sum of squares within
                    1e-6 relative of the float64 sum, from non-zero meters, at every width, filter kind and tail length
    no perturbation rows, bus and carried state of a metered render are those of the plain render
    invariance      meter bits do not depend on which outputs are requested or on the render mode
    inactive        inactive, never-active and padding entries keep their bits
    accumulation    K calls after one zeroing against the per-call meters
    time-split      a metered block takes the default path; plain blocks still take the time-split kernels
    edits           note-ons and note-off tables between metered renders
    non-finite      a cutoff swept past Nyquist: peak reads NaN / inf as the rows do, the sum is non-finite
    validation      null or misaligned meters change nothing; one meter without the other is refused
    launches        a metered render issues the launches of the same plain render
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import synth2_b200 as s2  # noqa: E402
from synth2_b200 import _lib  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402
from test_gpu_edits import SR, _bank  # noqa: E402

pytestmark = pytest.mark.gpu

FILTERS = (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP, s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP,
           s2.FILTER_FIRST_ORDER_LP, s2.FILTER_FIRST_ORDER_HP)
FRAMES = (1, 15, 16, 17, 64, 100, 4096, 4099)
SUM_SENTINEL = -1234.5
PEAK_SENTINEL = 0x00000123                      # a subnormal: any audible voice raises it


def _meters(V, sum_value=0.0, peak_bits=0, guard=0):
    """(sum_sq, peak, sum_buffer, peak_buffer): float64 / float32 device meters of V entries, views of buffers with
    `guard` extra entries after them.  Filled before it returns: a pipelined bank's streams do not wait for torch's."""
    sb = torch.full((V + guard,), sum_value, dtype=torch.float64, device="cuda")
    pb = torch.full((V + guard,), peak_bits, dtype=torch.int32, device="cuda").view(torch.float32)
    torch.cuda.synchronize()
    return sb[:V], pb[:V], sb, pb


def _rows(V, fr, fill=None):
    """A (V, fr) view of a device buffer whose row stride is fr rounded up to a multiple of 4 (the render's rule)."""
    cols = (fr + 3) & ~3
    buf = torch.empty((V, cols), device="cuda") if fill is None else torch.full((V, cols), fill, device="cuda")
    return buf[:, :fr]


def _ref(rows):
    """float64 sum of squares and magnitude bits of the peak of each row (device tensors)."""
    return rows.double().square().sum(dim=1), (rows.view(torch.int32) & 0x7fffffff).max(dim=1).values


def _bits(peak):
    return peak.view(torch.int32)


def _check(sum_sq, peak, prior_sum, prior_peak, sums, peaks, active, what):
    """Active voices: sum_sq within 1e-6 of prior + sums, relative to |prior| + sums (a negative prior may cancel the
    sum), peak bits = max(prior, peaks).  Others: unchanged."""
    want = prior_sum + sums
    act = torch.as_tensor(active, device="cuda")
    err = (sum_sq - want).abs()
    bound = 1e-6 * (prior_sum.abs() + sums) + 1e-300
    bad = act & ~(err <= bound)
    assert not bool(bad.any()), f"{what}: sum_sq off at voices {torch.nonzero(bad)[:8].flatten().tolist()}"
    want_pk = torch.maximum(prior_peak, peaks)
    badp = act & (_bits(peak) != want_pk)
    assert not bool(badp.any()), f"{what}: peak off at voices {torch.nonzero(badp)[:8].flatten().tolist()}"
    assert torch.equal(sum_sq[~act].view(torch.int64), prior_sum[~act].view(torch.int64)), f"{what}: inactive sum moved"
    assert torch.equal(_bits(peak)[~act], prior_peak[~act]), f"{what}: inactive peak moved"


# ------------------------------------------------------------------------------ 1. meters against the same call's rows

WIDTHS = (1, 7, 32, 33, 100, 2048, 65536)
ROWS_CASES = [(V, fk) for V in WIDTHS for fk in FILTERS]


@pytest.mark.parametrize("V,fk", ROWS_CASES, ids=[f"{V}v-filter{fk}" for V, fk in ROWS_CASES])
def test_meters_match_rows(V, fk):
    """Consecutive metered renders of every tail length from non-zero meters; each call's meters against its rows."""
    v = _bank(V, fk, V * 7 + fk)
    active = v["active"] != 0
    rng = np.random.default_rng(V + fk)
    rows = _rows(V, max(FRAMES))
    with s2.VoiceBank(v, SR, fk) as bank:
        for fr in FRAMES:
            prior_sum = torch.as_tensor(rng.uniform(0.0, 50.0, V), device="cuda")
            prior_peak = torch.as_tensor(rng.integers(0, 0x3f000000, V, dtype=np.int32), device="cuda")
            sum_sq, peak, _, _ = _meters(V)
            sum_sq.copy_(prior_sum)
            _bits(peak).copy_(prior_peak)
            torch.cuda.synchronize()
            out = rows[:, :fr]
            bank.render(fr, out, rows.stride(0), None, sum_sq, peak)
            bank.sync()
            sums, peaks = _ref(out)
            _check(sum_sq, peak, prior_sum, prior_peak, sums, peaks, active, f"{V} voices, filter {fk}, {fr} frames")


# ------------------------------------------------------------------------------ 2. no perturbation

@pytest.mark.parametrize("mode", [1, 2, 4, "ts"])
def test_metered_render_changes_no_output(mode):
    """Twin banks, one rendered plain and one metered: rows, bus and state bytes after every call.  A time-split bank's
    metered blocks take the default path, so its twin renders plain with time-split off."""
    V = 1000 if mode == "ts" else 4096
    fk = s2.FILTER_ONE_POLE if mode == "ts" else s2.FILTER_BIQUAD_LP
    v = _bank(V, fk, 41, late=mode == "ts")
    seq = (4096, 1000, 17, 2048, 4099)
    with s2.VoiceBank(v, SR, fk) as plain, s2.VoiceBank(v, SR, fk) as metered:
        if mode == "ts":
            metered.set_time_split(True)
        else:
            plain.set_pipeline(mode)
            metered.set_pipeline(mode)
        sum_sq, peak, _, _ = _meters(V)
        for fr in seq:
            got = [_rows(V, fr, float("nan")), torch.full((fr,), float("nan"), device="cuda")]
            want = [_rows(V, fr, float("nan")), torch.full((fr,), float("nan"), device="cuda")]
            torch.cuda.synchronize()
            plain.render(fr, want[0], want[0].stride(0), want[1])
            metered.render(fr, got[0], got[0].stride(0), got[1], sum_sq, peak)
            plain.sync()
            metered.sync()
            assert bool(torch.isfinite(want[0]).all())
            for name, a, b in zip(("rows", "bus"), got, want):
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{fr} frames: {name} differ"
            assert metered.get_state().tobytes() == plain.get_state().tobytes(), f"{fr} frames: state differs"
        if mode == "ts":
            assert metered.time_split_blocks == 0


# ------------------------------------------------------------------------------ 3. invariance

def _meter_run(v, fk, n_sub, outputs, seq):
    """Meters after the renders `seq` from zero; outputs = (rows, bus) requested alongside."""
    V = v.shape[0]
    sum_sq, peak, _, _ = _meters(V)
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        for fr in seq:
            rows = _rows(V, fr) if outputs[0] else None
            bus = torch.empty(fr, device="cuda") if outputs[1] else None
            bank.render(fr, rows, 0 if rows is None else rows.stride(0), bus, sum_sq, peak)
        bank.sync()
    return sum_sq.view(torch.int64).clone(), _bits(peak).clone()


def test_meter_bits_do_not_depend_on_outputs_or_mode():
    """65,536 voices: meters only, rows, bus, rows + bus, by one stream and by 2 and 4 voice ranges: the same bits."""
    V, fk = 65536, s2.FILTER_BIQUAD_LP
    v = bankgen.make_bank(V, 1 << 16, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE),
                          mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    seq = (4096, 4099, 100, 4096)
    base = _meter_run(v, fk, 1, (False, False), seq)
    assert bool((base[0] != 0).all()), "a voice rendered silence"
    for n_sub in (1, 2, 4):
        for outputs in ((False, False), (True, False), (False, True), (True, True)):
            if n_sub == 1 and outputs == (False, False):
                continue
            got = _meter_run(v, fk, n_sub, outputs, seq)
            what = f"{n_sub} ranges, rows={outputs[0]} bus={outputs[1]}"
            assert torch.equal(got[0], base[0]), f"{what}: sum_sq bits differ"
            assert torch.equal(got[1], base[1]), f"{what}: peak bits differ"


# ------------------------------------------------------------------------------ 4. inactive voices

@pytest.mark.parametrize("V,n_sub", [(33, 1), (1000, 1), (1000, 4)])
def test_inactive_voices_keep_their_entries(V, n_sub):
    """Sentinels in both arrays and past their end: never-active voices, voices a note-on batch turned off and the
    entries after the last voice keep them; active voices accumulate onto them."""
    fk = s2.FILTER_ONE_POLE
    v = _bank(V, fk, 5)
    off = np.flatnonzero(v["active"] != 0)[1::3].astype(np.uint32)
    d = v[off].copy()
    d["active"] = 0
    active = v["active"] != 0
    active[off] = False
    assert (v["active"] == 0).any() and off.size > 0
    guard = 16
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        bank.render(1000, None, 0, None)
        bank.set_voices(off, d)
        sum_sq, peak, sb, pb = _meters(V, SUM_SENTINEL, PEAK_SENTINEL, guard)
        prior_sum, prior_peak = sum_sq.clone(), _bits(peak).clone()
        torch.cuda.synchronize()
        rows = _rows(V, 2050)
        bank.render(2050, rows, rows.stride(0), None, sum_sq, peak)
        bank.sync()
    sums, peaks = _ref(rows)
    _check(sum_sq, peak, prior_sum, prior_peak, sums, peaks, active, f"{V} voices, {n_sub} ranges")
    sentinel = torch.tensor([SUM_SENTINEL], dtype=torch.float64).view(torch.int64).item()
    assert bool((sb.view(torch.int64)[V:] == sentinel).all()) and bool((_bits(pb)[V:] == PEAK_SENTINEL).all())
    assert bool((rows[torch.as_tensor(~active, device="cuda")] == 0).all())


# ------------------------------------------------------------------------------ 5. accumulation across calls

@pytest.mark.parametrize("n_sub", [1, 4])
def test_meters_accumulate_across_calls(n_sub):
    """K calls on one pair of meters against the same calls on a twin bank, each with freshly zeroed meters."""
    V, fk = 2048, s2.FILTER_BIQUAD_LP
    v = _bank(V, fk, 8)
    seq = (4096, 17, 4099, 1, 2048)
    acc_sum, acc_peak, _, _ = _meters(V)
    sums, peaks = [], []
    with s2.VoiceBank(v, SR, fk) as a, s2.VoiceBank(v, SR, fk) as b:
        a.set_pipeline(n_sub)
        b.set_pipeline(n_sub)
        for fr in seq:
            a.render(fr, None, 0, None, acc_sum, acc_peak)
            s, p, _, _ = _meters(V)
            b.render(fr, None, 0, None, s, p)
            sums.append(s)
            peaks.append(p)
        a.sync()
        b.sync()
    want = torch.stack(sums).sum(dim=0)
    assert bool(((acc_sum - want).abs() <= 1e-6 * want).all())
    assert torch.equal(_bits(acc_peak), torch.stack([_bits(p) for p in peaks]).max(dim=0).values)


# ------------------------------------------------------------------------------ 6. time-split

def test_metered_blocks_leave_the_time_split_path_alone():
    V, T = 1024, 4096
    voices = bankgen.make_bank(V, 1 << 20)
    active = voices["active"] != 0
    with s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE) as bank:
        bank.set_time_split(True)
        rows = torch.empty((V, T), device="cuda")
        for k in range(3):
            n0 = bank.time_split_blocks
            sum_sq, peak, _, _ = _meters(V)
            bank.render(T, rows, T, None, sum_sq, peak)
            bank.sync()
            assert bank.time_split_blocks == n0, "a metered block took the time-split kernels"
            sums, peaks = _ref(rows)
            _check(sum_sq, peak, torch.zeros_like(sum_sq), torch.zeros_like(_bits(peak)), sums, peaks, active,
                   f"time-split bank, block {k}")
            bank.render(T, rows, T, None)
            bank.sync()
            assert bank.time_split_blocks == n0 + 1, "a plain block did not take the time-split kernels"


# ------------------------------------------------------------------------------ 7. edits between metered renders

@pytest.mark.parametrize("n_sub", [1, 4])
def test_meters_follow_edits_between_renders(n_sub):
    """Note-on batches and note-off tables between metered renders: the meters keep the rows of those calls."""
    V, fk = 4096, s2.FILTER_BIQUAD_LP
    v = _bank(V, fk, 13)
    pool = _bank(64, fk, 14)
    rng = np.random.default_rng(15)
    sum_sq, peak, _, _ = _meters(V)
    want_sum = torch.zeros(V, dtype=torch.float64, device="cuda")
    want_peak = torch.zeros(V, dtype=torch.int32, device="cuda")
    everyone = np.ones(V, dtype=bool)
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        for k in range(6):
            fr = int(rng.choice([4096, 1000, 17, 2048]))
            rows = _rows(V, fr)
            bank.render(fr, rows, rows.stride(0), None, sum_sq, peak)
            bank.sync()
            s, p = _ref(rows)
            want_sum += s
            want_peak = torch.maximum(want_peak, p)
            _check(sum_sq, peak, torch.zeros_like(want_sum), torch.zeros_like(want_peak), want_sum, want_peak,
                   everyone, f"{n_sub} ranges, after render {k}")
            if k % 2 == 0:
                idx = rng.choice(V, 200, replace=False).astype(np.uint32)
                d = pool[rng.integers(0, 64, idx.size)].copy()
                d["active"] = rng.random(idx.size) < 0.8
                d["frame_offset"] = rng.integers(0, 20000, idx.size)
                bank.set_voices(idx, d)
            else:
                st = bank.get_state()
                bank.set_releases((st["frame_offset"] + rng.integers(0, 3000, V)).astype(np.uint32))


# ------------------------------------------------------------------------------ 8. non-finite output

@pytest.mark.parametrize("fk", [s2.FILTER_BIQUAD_LP, s2.FILTER_BIQUAD_HP])
def test_non_finite_rows_show_in_the_meters(fk):
    """Cutoffs opened by the mod envelope to up to 8x 6 kHz, far past Nyquist: the filter state overflows to inf and
    then NaN (ordinary float arithmetic).  Peak bits are those of the rows; the sum of squares is non-finite."""
    V, T = 256, 4099
    v = bankgen.make_bank(V, 1 << 16, mod_to_lpf_choices=(0.0, 3.0))
    v["lpf_freq_hz"] = np.linspace(200.0, 6000.0, V, dtype=np.float32)
    v["mod_decay_ms"] = 1000.0
    v["mod_sustain"] = 1.0
    active = v["active"] != 0
    with s2.VoiceBank(v, SR, fk) as bank:
        sum_sq, peak, _, _ = _meters(V)
        rows = _rows(V, T)
        for k in range(4):
            bank.render(T, rows, rows.stride(0), None, sum_sq, peak)
            bank.sync()
            if not bool(torch.isfinite(rows).all()):
                break
    sums, peaks = _ref(rows)
    bad = ~torch.isfinite(rows).all(dim=1)
    assert bool(bad.any()), "no voice blew up"
    assert bool((_bits(peak)[bad] == peaks[bad]).all()), "peak bits differ from the rows' on non-finite voices"
    assert bool((~torch.isfinite(sum_sq[bad])).all()), "a non-finite voice has a finite sum of squares"
    assert bool(torch.isnan(peak[torch.isnan(rows).any(dim=1)]).all())


# ------------------------------------------------------------------------------ 9. validation

@pytest.mark.parametrize("n_sub", [1, 4])
def test_invalid_meters_change_nothing(n_sub):
    V, T, fk = 1000, 1024, s2.FILTER_BIQUAD_LP
    v = _bank(V, fk, 17)
    lib = s2.lib()
    sb = torch.zeros(V + 2, dtype=torch.float64, device="cuda")
    pb = torch.zeros(V + 2, dtype=torch.float32, device="cuda")
    rows = torch.full((V, T), float("nan"), device="cuda")
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        bank.render(T, None, 0, None)
        bank.sync()
        st = bank.get_state()
        s, p = sb.data_ptr(), pb.data_ptr()
        cases = [(None, p), (s, None), (None, None), (s + 4, p), (s + 1, p), (s, p + 2), (s, p + 1)]
        n0 = lib.s2_launch_count()
        for cs, cp in cases:
            rc = lib.s2_bank_render_metered(bank._h, T, _lib.ptr(rows), T, None,
                                            None if cs is None else C.c_void_p(cs), None if cp is None else C.c_void_p(cp))
            assert rc == _lib.S2_ERR_INVALID, (cs, cp)
        assert lib.s2_bank_render_metered(None, T, None, 0, None, C.c_void_p(s), C.c_void_p(p)) == _lib.S2_ERR_INVALID
        assert lib.s2_launch_count() == n0, "an invalid call launched a kernel"
        bank.sync()
        assert bank.get_state().tobytes() == st.tobytes(), "an invalid call moved the state"
        assert bool(torch.isnan(rows).all()) and bool((sb == 0).all()) and bool((pb == 0).all())
        with pytest.raises(ValueError):
            bank.render(T, None, 0, None, sb[:V], None)
        with pytest.raises(ValueError):
            bank.render(T, None, 0, None, None, pb[:V])
        with pytest.raises(ValueError):
            bank.render(T, None, 0, None, pb[:V], sb[:V])           # dtypes swapped
        with pytest.raises(ValueError):
            bank.render(T, None, 0, None, sb, pb)                   # V + 2 entries
        assert lib.s2_launch_count() == n0
        bank.sync()
        assert bank.get_state().tobytes() == st.tobytes()


# ------------------------------------------------------------------------------ 10. launch counts

def _launches(fn, *args):
    n0 = s2.lib().s2_launch_count()
    fn(*args)
    return s2.lib().s2_launch_count() - n0


LAUNCH_CASES = [(V, mode) for V in (1, 33, 2048, 65536) for mode in (1, 2, 4, 8, "ts") if not (mode == "ts" and V > 16384)]


@pytest.mark.parametrize("V,mode", LAUNCH_CASES)
def test_metered_render_launches(V, mode):
    """The same launches as the plain render, with and without rows and bus.  A time-split bank's metered blocks are
    default-path blocks: they count as the plain render with time-split off."""
    T = 4096
    voices = bankgen.make_bank(V, 1 << 20)
    sum_sq, peak, _, _ = _meters(V)
    rows = torch.empty((V, T), device="cuda")
    bus = torch.empty(T, device="cuda")
    with s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE) as bank:
        if mode != "ts":
            bank.set_pipeline(mode)
        for r, b in ((None, None), (rows, None), (None, bus), (rows, bus)):
            stride = T if r is not None else 0
            if mode == "ts":
                bank.set_time_split(False)
            plain = _launches(bank.render, T, r, stride, b)
            if mode == "ts":
                bank.set_time_split(True)
            metered = _launches(bank.render, T, r, stride, b, sum_sq, peak)
            assert metered == plain, (r is not None, b is not None)
        bank.sync()
