"""The mono bus (`d_bus_out` of s2_bank_render, the host copy of s2_bank_render_bus_host[_async]): what the library
plays, checked against exact references at every bank width and render mode.

- Exact-sum banks (busref.exact_bank): every sample sits on the 2^-14 grid and every partial sum is exact, so the
  bus must equal the float64 sum of the rows bit for bit whatever the summation tree.  Every bus buffer starts as
  NaN and sits 16 bytes into a NaN guard, so a bus that is not written, or written outside [0, frames), fails.
- Banks of <= 32 voices: the bus is the reference's sequential sum in voice order (synth.rs:176-202), in every
  mode, compared with tobytes() so that the sign of a zero counts.
- Realistic wide banks: within the error bound of the documented trees (busref.bus_depth), and bit-identical
  across renders from one state and across the pipelined voice ranges.
"""
import numpy as np
import pytest

import oracle
import synth2_b200 as s2
from busref import (GRID, advance, assert_bus_within_bound, closed_bus, closed_form, closed_rows, exact_bank,
                    reference_order_bus)
from synth2_b200 import bankgen

SR = 48000
WIDTHS = [1, 31, 32, 33, 65, 1000, 16352, 16384, 16385, 65536]   # 16,352 = 511 warps; 16,384 the first wide bank
MODES = ["default", "pipe2", "pipe3", "pipe4", "pipe8", "host", "time_split"]
# frames per call.  X16: every call a multiple of 16, growing and shrinking, so that the wide reduction's frame-group
# counters are used for the first time (8,192 after 4,096) and again after their reset, and every scratch buffer
# grows while earlier calls are still queued.  TAIL: scalar-path tail frames (17, 100, 4,100 frames; 4,100 % 4 == 0
# but not % 128), for tail-safe banks.  BIG: more 128-frame groups than the wide reduction has counters.
X16_SEQ = [64, 128, 4096, 8192, 4096, 128, 8192, 1024, 4096]
TAIL_SEQ = [1, 17, 100, 4100, 64, 4096]
BIG = 131200


# ------------------------------------------------------------------------------ the construction, on the CPU

@pytest.mark.parametrize("tail_safe", [False, True])
def test_exact_construction_matches_the_oracle(tail_safe):
    """The exact banks as the oracle renders them: every sample on the 2^-14 grid, the x16 frames equal to the
    closed form bit for bit, the scalar tail frames equal to it in magnitude.  A mistake in the construction fails
    here, on any machine, rather than as a wrong bus on the GPU."""
    v = exact_bank(400, 5 + tail_safe, tail_safe=tail_safe, span=30000)
    st = oracle.bank_init_states(v)
    n0 = v["frame_offset"].astype(np.int64)
    seq = [4096, 1000, 17, 4100, 1, 63, 64, 8192] if tail_safe else [4096, 1024, 64, 8192, 16, 128]
    released = silent_neg_zero = 0
    for fr in seq:
        rows, _ = oracle.bank_render(v, st, SR, s2.FILTER_ONE_POLE, fr, want_bus=False, nthreads=8)
        q = rows.astype(np.float64) / GRID
        assert np.all(q == np.round(q)) and np.all(np.abs(q) <= 255), fr
        val, stop = closed_form(v, n0, fr)
        want = closed_rows(val, stop, fr)
        x = fr - fr % 16
        assert np.array_equal(rows[:, :x], want[:, :x]), fr
        assert np.array_equal(np.abs(rows[:, x:]), np.abs(want[:, x:])), fr
        released += int(np.sum((stop > 0) & (stop < fr)))
        silent_neg_zero += int(np.sum(np.signbit(rows[rows == 0])))
        n0 = advance(v, n0, fr)
    assert np.array_equal(st["frame_offset"], n0.astype(np.uint32))
    assert released > 50 and silent_neg_zero > 0      # note-offs land inside calls; released voices give -0.0
    assert int(np.sum(v["amp_sustain"].astype(np.float64) * 2.0 ** 40)) < (1 << 24)


# ------------------------------------------------------------------------------ GPU

torch = pytest.importorskip("torch")


def _exact(n, seed, tail_safe):
    v = exact_bank(n, seed, tail_safe=tail_safe)
    # voice 0 sounds with a negative gain and is released during the first calls: its silent frames are -0.0
    v[0]["active"] = 1
    v[0]["osc_gain"] = -(2.0 ** 26)
    v[0]["release_offset"] = int(v[0]["frame_offset"]) + 3000
    return v


def _bus_bits(x):
    return np.asarray(x, dtype=np.float32).view(np.uint32)


def _apply_mode(bank, mode):
    if mode.startswith("pipe"):
        bank.set_pipeline(int(mode[4:]))
    elif mode == "time_split":
        bank.set_time_split(True)


def _run(bank, mode, seq, with_rows, big=None):
    """Renders `seq` back to back (no host sync in between, except that the host modes synchronise by nature) and
    returns, per call, (frames, rows tensor or None, guarded bus) after one sync.  Rows have a padded stride."""
    V = bank.n_voices
    calls = []
    for fr in seq + ([big] if big else []):
        rows = None
        if with_rows and fr != big:
            rows = torch.full((V, ((fr + 3) & ~3) + 4), float("nan"), device="cuda", dtype=torch.float32)
        if mode == "host":
            bus = np.full(fr + 8, np.nan, dtype=np.float32)
        else:
            bus = torch.full((fr + 8,), float("nan"), device="cuda", dtype=torch.float32)
        calls.append((fr, rows, bus))
    torch.cuda.synchronize()             # the NaN fills are done before any of the bank's streams writes
    for fr, rows, bus in calls:
        stride = 0 if rows is None else rows.stride(0)
        if mode == "host":
            bank.render_bus_host(fr, rows, stride, out=bus[4:4 + fr])
        else:
            bank.render(fr, rows, stride, bus[4:4 + fr])
    bank.sync()
    out = []
    for fr, rows, bus in calls:
        b = bus if mode == "host" else bus.cpu().numpy()
        assert np.all(np.isnan(b[:4])) and np.all(np.isnan(b[4 + fr:])), f"bus written outside [0, {fr})"
        out.append((fr, rows, b[4:4 + fr].copy()))
    return out


def _check_exact_call(v, n0, fr, rows, bus, what):
    """Rows (when given) against the closed form; the bus against the exact sum.  Returns the expected bus."""
    val, stop = closed_form(v, n0, fr)
    x = fr - fr % 16
    if rows is not None:
        assert bool(torch.isnan(rows[:, fr:]).all()), f"{what}: row written past frames"
        r = rows[:, :fr]
        ar = torch.arange(fr, device="cuda")
        want = torch.where(ar[None, :] < torch.as_tensor(stop, device="cuda")[:, None],
                           torch.as_tensor(val, device="cuda")[:, None], torch.zeros((), device="cuda"))
        assert torch.equal(r[:, :x], want[:, :x]), f"{what}: x16 rows differ from the closed form"
        assert torch.equal(r[:, x:].abs(), want[:, x:].abs()), f"{what}: tail rows differ from the closed form"
        expect = (r.double().sum(dim=0).cpu().numpy() + 0.0).astype(np.float32)   # exact: on the grid
        if x == fr:
            assert np.array_equal(_bus_bits(expect), _bus_bits(closed_bus(val, stop, fr)))
    else:
        assert x == fr, "a bus-only tail call needs its expectation from a call with rows"
        expect = closed_bus(val, stop, fr)
    assert np.array_equal(_bus_bits(bus), _bus_bits(expect)), (
        f"{what}: bus differs from the exact sum at {int(np.sum(_bus_bits(bus) != _bus_bits(expect)))} of {fr} frames")
    return expect


CASES = [(w, m) for w in WIDTHS for m in MODES if not (m == "time_split" and w > 16384)]


@pytest.mark.gpu
@pytest.mark.parametrize("width,mode", CASES, ids=[f"{w}-{m}" for w, m in CASES])
def test_exact_bus(width, mode):
    """Exact banks at every width and mode: a call sequence with rows (padded stride), then the same calls again
    from the same state without rows (time-split then falls back to the default path), and one call of more
    frame groups than the wide reduction has counters.  Bus bit-exact after every call."""
    for tail_safe, seq in ((False, X16_SEQ), (True, TAIL_SEQ)):
        v = _exact(width, 1000 + width + 7 * tail_safe, tail_safe)
        with s2.VoiceBank(v, SR, s2.FILTER_ONE_POLE) as bank:
            _apply_mode(bank, mode)
            state0 = bank.get_state()
            ts0 = bank.time_split_blocks
            first = _run(bank, mode, seq, True, big=None if tail_safe else BIG)
            if mode == "time_split":
                assert bank.time_split_blocks - ts0 == sum(1 for fr in seq if fr % 1024 == 0)
            bank.set_state(state0)
            ts1 = bank.time_split_blocks
            second = _run(bank, mode, seq, False)
            assert bank.time_split_blocks == ts1            # no rows: the time-split path is not taken
        n0 = v["frame_offset"].astype(np.int64)
        buses = []
        for i, (fr, rows, bus) in enumerate(first):
            buses.append(_check_exact_call(v, n0, fr, rows, bus, f"{mode} call {i} ({fr} frames, rows)"))
            n0 = advance(v, n0, fr)
        for i, (fr, _, bus) in enumerate(second):
            assert np.array_equal(_bus_bits(bus), _bus_bits(buses[i])), f"{mode} call {i} ({fr} frames, bus only)"


@pytest.mark.gpu
def test_exact_bus_mode_switches():
    """Default -> pipeline 4 -> pipeline 2 -> default on one wide bank, and time-split on -> off on a narrow one,
    with a bus on every call and the scratch buffers growing across the switches."""
    for width, plan in ((65536, [("default", 128), ("pipe4", 4096), ("pipe4", 8192), ("pipe2", 128),
                                 ("pipe2", 8192), ("default", 4096), ("default", 8192)]),
                        (16385, [("pipe4", 8192), ("default", 4096), ("pipe8", 4096), ("default", 128)]),
                        (16384, [("time_split", 4096), ("time_split", 8192), ("off", 4096), ("off", 128),
                                 ("time_split", 1024)])):
        v = _exact(width, 77 + width, False)
        n0 = v["frame_offset"].astype(np.int64)
        with s2.VoiceBank(v, SR, s2.FILTER_ONE_POLE) as bank:
            for i, (mode, fr) in enumerate(plan):
                if mode == "off":
                    bank.set_time_split(False)
                elif mode.startswith("pipe"):
                    bank.set_pipeline(int(mode[4:]))
                elif mode == "default":
                    bank.set_pipeline(1)
                else:
                    bank.set_time_split(True)
                ts0 = bank.time_split_blocks
                (_, rows, bus), = _run(bank, "default", [fr], True)
                assert bank.time_split_blocks - ts0 == (1 if mode == "time_split" else 0)
                _check_exact_call(v, n0, fr, rows, bus, f"{width} voices, step {i} ({mode}, {fr} frames)")
                n0 = advance(v, n0, fr)


@pytest.mark.gpu
def test_exact_bus_bench_e2e_loop():
    """bench.py's e2e loop at full width: pipeline 4, a note-off table uploaded before every step (a new one each
    step here), render + mix + copy of the mix into one of two pinned host buffers, the host consuming step i - 1
    after enqueuing step i.  Every host bus bit-exact."""
    V, T, N = 65536, 4096, 12
    v = _exact(V, 4242, False)
    rng = np.random.default_rng(9)
    stream = torch.cuda.current_stream()
    ring = [torch.empty((V, T), device="cuda") for _ in range(2)]
    bus_host = [torch.empty(T, dtype=torch.float32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    n0 = v["frame_offset"].astype(np.int64)
    tables, expect = [], []
    rel = v["release_offset"].astype(np.int64)
    for i in range(N):
        rel = rel.copy()
        pick = rng.random(V) < 0.05
        rel[pick] = np.where(rng.random(V) < 0.8, n0 + rng.integers(-100, T + 100, V), 0xFFFFFFFF)[pick]
        rel = np.clip(rel, 0, 0xFFFFFFFF)
        tables.append(torch.from_numpy(rel.astype(np.uint32).view(np.int32)).pin_memory())
        val, stop = closed_form(v, n0, T, release=rel)
        expect.append(closed_bus(val, stop, T))
        n0 = advance(v, n0, T)
    got = [None] * N
    with s2.VoiceBank(v, SR, s2.FILTER_ONE_POLE, stream=stream) as bank:
        bank.set_pipeline(4)
        for i in range(N):
            bus_host[i & 1].fill_(float("nan"))
            bank.set_releases(tables[i])
            bank.render_bus_host_async(T, bus_host[i & 1], ring[i & 1], T)
            done[i & 1].record(stream)
            if i > 0:
                done[(i - 1) & 1].synchronize()
                got[i - 1] = bus_host[(i - 1) & 1].numpy().copy()
        done[(N - 1) & 1].synchronize()
        got[N - 1] = bus_host[(N - 1) & 1].numpy().copy()
        bank.join(stream)
        stream.synchronize()
    for i in range(N):
        assert np.array_equal(_bus_bits(got[i]), _bus_bits(expect[i])), f"step {i}"
    assert len({e.tobytes() for e in expect}) == N          # the steps' buses differ


@pytest.mark.gpu
def test_exact_master_bus_one_rank():
    """s2_bank_reduce_bus on a one-rank communicator after a wide pipelined render: master = the exact sum."""
    from synth2_b200.shard import MasterBus
    V, T = 65536, 4096
    v = _exact(V, 31337, False)
    val, stop = closed_form(v, v["frame_offset"], T)
    with s2.VoiceBank(v, SR, s2.FILTER_ONE_POLE) as bank:
        bank.set_pipeline(4)
        bus = torch.full((T,), float("nan"), device="cuda")
        master = torch.full((T,), float("nan"), device="cuda")
        torch.cuda.synchronize()
        bank.render(T, None, 0, bus)
        with MasterBus(0, 1, 0) as comm:
            comm.reduce(bank, bus, master, root=0, stream=torch.cuda.current_stream())
            torch.cuda.synchronize()
    assert np.array_equal(_bus_bits(master.cpu().numpy()), _bus_bits(closed_bus(val, stop, T)))


# ------------------------------------------------------------------------------ <= 32 voices: the reference's order

NARROW_MODES = ["default", "bus_only", "pipe2", "pipe4", "host", "host_async", "time_split"]
NARROW_SEQ = [4096, 4096, 1024, 2048, 100, 17]


def _narrow_bank(V, filter_kind, seed):
    sweep = bankgen.MOD_TO_LPF_BIQUAD if filter_kind == s2.FILTER_BIQUAD_LP else bankgen.MOD_TO_LPF_ONE_POLE
    v = bankgen.make_bank(V, 8192, first_voice=seed * 64, kinds=(s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE,
                                                                   s2.OSC_SINE), mod_to_lpf_choices=sweep)
    v["osc_gain"] = np.array([0.0, 0.5, 1.0], np.float32)[np.arange(V) % 3]
    v["amp_attack_ms"] = np.minimum(v["amp_attack_ms"], 40.0)
    v["amp_decay_ms"] = np.minimum(v["amp_decay_ms"], 40.0)
    v["amp_release_ms"] = 5.0 + (np.arange(V) % 5) * 5.0     # released at 6,144: every voice ends by frame 7,344
    if V > 2:
        v["release_offset"][1] = s2.NO_RELEASE
    return v


def _narrow_render(v, filter_kind, mode):
    """Renders NARROW_SEQ in `mode`; returns [(rows [V, fr] numpy or None, bus numpy)] and the time-split count."""
    V = v.shape[0]
    stream = torch.cuda.current_stream()
    out = []
    with s2.VoiceBank(v, SR, filter_kind, stream=stream) as bank:
        if mode in ("pipe2", "pipe4", "host_async"):
            bank.set_pipeline(4 if mode == "pipe4" else 2)
        if mode == "time_split":
            bank.set_time_split(True)
        for fr in NARROW_SEQ:
            stride = ((fr + 3) & ~3) + 12
            rows = None if mode == "bus_only" else torch.full((V, stride), float("nan"), device="cuda")
            stride = 0 if rows is None else stride
            if mode == "host":
                bus = bank.render_bus_host(fr, rows, stride)
            elif mode == "host_async":
                pinned = torch.full((fr,), float("nan")).pin_memory()
                torch.cuda.synchronize()
                bank.render_bus_host_async(fr, pinned, rows, stride)
                bank.join(stream)
                stream.synchronize()
                bus = pinned.numpy().copy()
            else:
                b = torch.full((fr,), float("nan"), device="cuda")
                torch.cuda.synchronize()
                bank.render(fr, rows, stride, b)
                bank.sync()
                bus = b.cpu().numpy()
            out.append((None if rows is None else rows[:, :fr].cpu().numpy(), bus))
        n_ts = bank.time_split_blocks
    return out, n_ts


@pytest.mark.gpu
@pytest.mark.parametrize("mode", NARROW_MODES)
@pytest.mark.parametrize("filter_kind", [s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP])
@pytest.mark.parametrize("V", [1, 2, 7, 32])
def test_narrow_bus_is_the_reference_sum(V, filter_kind, mode):
    """Banks of up to one warp: the bus is acc = 0.0f; acc = acc + row[v] in voice order, bit for bit (tobytes:
    -0.0 from a released voice must come out as +0.0, as the reference's 0.0 + x does), in every mode."""
    v = _narrow_bank(V, filter_kind, 3 + V)
    got, n_ts = _narrow_render(v, filter_kind, mode)
    if mode == "bus_only":
        rows_of, _ = _narrow_render(v, filter_kind, "default")
        rows_of = [r for r, _ in rows_of]
    else:
        rows_of = [r for r, _ in got]
    assert n_ts == (sum(1 for fr in NARROW_SEQ if fr % 1024 == 0) if mode == "time_split" else 0)
    neg_zero = 0
    for i, ((_, bus), rows) in enumerate(zip(got, rows_of)):
        assert np.all(np.isfinite(rows)), i
        want = reference_order_bus(rows)
        assert bus.tobytes() == want.tobytes(), (
            f"call {i}: {int(np.sum(bus.view(np.uint32) != want.view(np.uint32)))} of {bus.size} frames differ")
        neg_zero += int(np.sum(np.signbit(rows[rows == 0])))
    assert neg_zero > 0                  # the case that tells a copy of the row from a sum that starts at +0.0


# ------------------------------------------------------------------------------ realistic wide banks

@pytest.mark.gpu
@pytest.mark.parametrize("V", [16384, 65536])
@pytest.mark.parametrize("filter_kind", [s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP])
def test_wide_bus_bound_and_determinism(filter_kind, V):
    """Config-3-like banks (and their one-pole twins): on every call the bus is within gamma_d * sum|rows| of the
    exact sum of the rows the same render produced (under 1 at 65,536 voices: a missing or doubled voice is 1-3),
    bit-identical between two renders from one state, and bit-identical across the default path and pipelines of
    2, 3, 4 and 8 voice ranges.  Time-split blocks (16,384 voices) within their own bound."""
    sweep = bankgen.MOD_TO_LPF_BIQUAD if filter_kind == s2.FILTER_BIQUAD_LP else bankgen.MOD_TO_LPF_ONE_POLE
    v = bankgen.make_bank(V, 16384, mod_to_lpf_choices=sweep)
    v["active"][5::97] = 0
    seq = [4096, 128, 8192, 100]
    modes = ["default", "again", "pipe2", "pipe3", "pipe4", "pipe8"] + (["time_split"] if V <= 16384 else [])
    buses = {}
    with s2.VoiceBank(v, SR, filter_kind) as bank:
        state0 = bank.get_state()
        for mode in modes:
            bank.set_state(state0)
            bank.set_pipeline(int(mode[4:]) if mode.startswith("pipe") else 1)
            if mode == "time_split":
                bank.set_time_split(True)
            ts0 = bank.time_split_blocks
            calls = _run(bank, "default", seq, True)
            assert bank.time_split_blocks - ts0 == (2 if mode == "time_split" else 0)
            for i, (fr, rows, bus) in enumerate(calls):
                path = "time_split" if mode == "time_split" and fr % 1024 == 0 else "default"
                assert_bus_within_bound(bus, rows[:, :fr], V, path, f"{mode} call {i} ({fr} frames)")
            buses[mode] = [b for _, _, b in calls]
            del calls
    for mode in modes[1:]:
        if mode == "time_split":
            continue
        for i in range(len(seq)):
            assert buses[mode][i].tobytes() == buses["default"][i].tobytes(), f"{mode} call {i} differs from default"
