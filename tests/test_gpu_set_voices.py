"""Bulk note-on, s2_bank_set_voices: the same effect as set_voice called for each entry in order, applied on the GPU
without waiting for the bank's renders.

    same bytes      a batch against the same set_voice calls on a twin bank: rows, bus, phase trace and state byte for
                    byte, at every width and render mode
    call order      seeded scripts that mix batches with note-off tables, release_voice, set_voice, set_state, traces
                    and mode changes, against the oracle model of test_gpu_edits (pipelined runs byte for byte with the
                    one-stream run, time-split runs within tolerance with the predicted time-split blocks)
    re-patch        a batch over the whole bank equals a new bank made from the same descriptions, also when the
                    staging buffers grow while pipelined renders are in flight
    validation      a bad entry anywhere changes nothing
    launches        one scatter per voice range that receives entries, none for an empty batch
    no wait         the call returns while the bank's stream is still busy
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import synth2_b200 as s2  # noqa: E402
from synth2_b200 import _lib  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402
from test_gpu_edits import (FRAMES, FRAMES_TS, RENDERS, SR, _bank, _fresh, _Model, _release_op,  # noqa: E402
                            _set_voice_op, _sweep, _synthetic_state, _table_op, check_run, compare_runs, describe)

pytestmark = pytest.mark.gpu


def _launches(fn, *args):
    n0 = s2.lib().s2_launch_count()
    fn(*args)
    return s2.lib().s2_launch_count() - n0


def _ranges(V, n_sub):
    """Non-empty voice ranges of a bank of V voices cut into n_sub ranges of whole 64-slot groups."""
    groups = -(-V // 64)
    bounds = [min(groups * k // n_sub * 64, V) for k in range(n_sub + 1)]
    return sum(1 for k in range(n_sub) if bounds[k] < bounds[k + 1])


# ------------------------------------------------------------------------------ batches

def _entry(rng, m, i, pool, fk, late):
    """One note-on for voice i, applied to the model: a fresh note, a deactivation, an oscillator kind change (to or
    from sine) or a cutoff follower turned into a resting voice (or back)."""
    form = str(rng.choice(["fresh", "fresh", "deactivate", "kind", "follower"]))
    if form == "fresh":
        d = _fresh(rng, pool, late)
    else:
        d = m.d[i:i + 1].copy()
        d["frame_offset"] = m.s["frame_offset"][i]
        if form == "deactivate":
            d["active"] = 0
        elif form == "kind":
            d["active"] = 1
            d["osc_kind"] = s2.OSC_SINE if d["osc_kind"][0] != s2.OSC_SINE else int(rng.integers(0, 3))
        else:
            d["active"] = 1
            d["mod_env_to_lpf_freq"] = 0.0 if d["mod_env_to_lpf_freq"][0] != 0.0 else _sweep(fk)[1]
    m.set_voice(i, d)
    return d[0]


def _batch(rng, m, pool, fk, late, form, size=None):
    """(indices, descriptions) of one batch, applied to the model in entry order.
    spread: random voices with repeats; all: every voice, in a random order; one: a single voice 1-3 times;
    pitchmod: spread, plus an active voice whose pitch follows the mod envelope."""
    V = m.d.shape[0]
    if form == "all":
        idx = rng.permutation(V)
    elif form == "one":
        idx = np.full(int(rng.integers(1, 4)), int(rng.integers(V)))
    else:
        k = size or int(rng.integers(2, min(V, 40) + 2))
        idx = rng.integers(0, V, k)
        idx = np.concatenate([idx, rng.choice(idx, max(1, k // 5))])          # repeated indices
        rng.shuffle(idx)
    descs = np.zeros(idx.size, dtype=s2.VOICE_DESC)
    for j, i in enumerate(map(int, idx)):
        descs[j] = _entry(rng, m, i, pool, fk, late)
    if form == "pitchmod":
        i = int(rng.integers(V))
        d = _fresh(rng, pool, late)
        d["mod_env_to_osc_freq"] = 0.5
        m.set_voice(i, d)
        idx = np.append(idx, i)
        descs = np.append(descs, d)
    return idx.astype(np.uint32), descs


# ------------------------------------------------------------------------------ 1. same bytes as set_voice in order

def _twin_run(v, fk, mode, batches, batched, F):
    """Render, batch 1, render, batch 2, render, trace; returns device rows / buses / trace, state, time-split blocks."""
    V = v.shape[0]
    rows = [torch.full((V, F), float("nan"), device="cuda") for _ in range(3)]
    buses = [torch.full((F,), float("nan"), device="cuda") for _ in range(3)]
    phase = torch.full((V, 1000), float("nan"), device="cuda")
    torch.cuda.synchronize()
    with s2.VoiceBank(v, SR, fk) as bank:
        if mode == "ts":
            bank.set_time_split(True)
        else:
            bank.set_pipeline(mode)
        bank.render(F, rows[0], F, buses[0])
        for k, (idx, descs) in enumerate(batches):
            if batched:
                bank.set_voices(idx, descs)
            else:
                for i, d in zip(idx, descs):
                    bank.set_voice(int(i), d)
            bank.render(F, rows[k + 1], F, buses[k + 1])
        bank.trace_phase(1000, phase)
        bank.sync()
        st = bank.get_state()
        ts = bank.time_split_blocks
    torch.cuda.synchronize()
    return rows + buses + [phase], st, ts


WIDTHS = (1, 7, 32, 33, 1000, 4096, 65536)
MODES = (1, 2, 3, 4, 8, "ts")
SAME = [(V, mode, fk) for V in WIDTHS for mode in MODES for fk in (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP)
        if not (mode == "ts" and V > 16384)] + \
       [(1000, 1, fk) for fk in (s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP, s2.FILTER_FIRST_ORDER_LP,
                                 s2.FILTER_FIRST_ORDER_HP)]


@pytest.mark.parametrize("V,mode,fk", SAME, ids=[f"{V}v-{'ts' if m == 'ts' else f'pipe{m}'}-filter{fk}"
                                                for V, m, fk in SAME])
def test_same_bytes_as_sequential_set_voice(V, mode, fk):
    """Two seeded batches (repeated indices, deactivations, kind changes to and from sine, followers turned resting)
    through set_voices on one bank and through the same set_voice calls in order on its twin."""
    seed = V * 31 + (0 if mode == "ts" else mode) * 7 + fk
    rng = np.random.default_rng(seed)
    late = mode == "ts"
    v = _bank(V, fk, seed, late=late)
    pool = _bank(64, fk, 60000 + seed, late=late)
    m = _Model(v, fk)
    size = max(3, V // 50)
    batches = [_batch(rng, m, pool, fk, late, "spread", size) for _ in range(2)]
    F = 2048
    got, got_st, got_ts = _twin_run(v, fk, mode, batches, True, F)
    want, want_st, want_ts = _twin_run(v, fk, mode, batches, False, F)
    names = ["rows 0", "rows 1", "rows 2", "bus 0", "bus 1", "bus 2", "phase trace"]
    for name, a, b in zip(names, got, want):
        assert bool(torch.isfinite(b).all()), f"{name}: not rendered"
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{name} differs from sequential set_voice"
    assert got_st.tobytes() == want_st.tobytes(), "state differs from sequential set_voice"
    assert got_ts == want_ts
    if mode == "ts":
        assert got_ts >= 1, "no block took the time-split path"


# ------------------------------------------------------------------------------ 2. call order against the oracle model

HAZARDS = ("table-batch", "table-batch-table", "batch-table", "two-batches", "batch-all-ranges", "batch-one-range",
           "batch-then-edit", "pitchmod")


def _render_op(rng, m, family, ts_on):
    call = str(rng.choice(["render", "render", "host", "async"]))
    fr = int(rng.choice(FRAMES_TS if family == "ts" else FRAMES))
    op = {"op": call, "frames": fr}
    if call == "render":
        op["rows"], op["bus"] = [(True, False), (False, True), (True, True), (True, True)][int(rng.integers(4))]
    else:
        op["rows"], op["bus"] = bool(rng.random() < 0.75), True
    if family == "ts":
        op["rows"] = True                  # time-split blocks need the rows
    op["ts"] = int(ts_on and op["rows"] and m.ts_block(fr))
    op["expect"] = m.render(fr)
    return op


def _trace_op(rng, m):
    fr = int(rng.choice([17, 1000, 2048]))
    return {"op": "trace", "frames": fr, "rows": False, "bus": False, "ts": 0, "expect": m.render(fr)}


def _batch_op(rng, m, pool, fk, late, form):
    idx, descs = _batch(rng, m, pool, fk, late, form)
    return {"op": "set_voices", "form": form, "idx": idx, "descs": descs}


def make_batch_script(seed, V, fk, family):
    """(voices, ops): every hazard of HAZARDS once, in a seeded order, each followed by a render, with other edits,
    traces, checkpoints and mode changes between them."""
    rng = np.random.default_rng(seed)
    late = family == "ts"
    v = _bank(V, fk, seed, late=late)
    pool = _bank(64, fk, 50000 + seed, late=late)
    m = _Model(v, fk)
    ts_on = family == "ts"
    ops = [{"op": "mode", "ts": True} if ts_on else {"op": "mode", "pipe": int(rng.choice([2, 3, 4, 8]))}]
    recent, checkpoints = [], []
    batch = lambda form="spread": _batch_op(rng, m, pool, fk, late, form)   # noqa: E731
    for hz in rng.permutation(HAZARDS):
        if hz == "table-batch":
            ops += [_table_op(rng, m), batch()]
        elif hz == "table-batch-table":
            ops += [_table_op(rng, m), batch(), _table_op(rng, m)]
        elif hz == "batch-table":
            ops += [batch(), _table_op(rng, m)]
        elif hz == "two-batches":
            ops += [batch(), batch()]
        elif hz == "batch-all-ranges":
            ops += [batch("all")]
        elif hz == "batch-one-range":
            ops += [_table_op(rng, m), batch("one")]
        elif hz == "pitchmod":
            ops += [batch("pitchmod")]
        else:
            ops.append(batch())
            edit = str(rng.choice(["set_voice", "release", "state", "trace", "mode", "checkpoint"]))
            if edit == "set_voice":
                ops.append(_set_voice_op(rng, m, pool, fk, late, recent))
            elif edit == "release":
                ops.append({"op": "release", "idx": [int(i) for i in ops[-1]["idx"][:3]]})
                for i in ops[-1]["idx"]:
                    m.release_voice(i)
            elif edit == "state":
                ops.append(_synthetic_state(rng, m))
            elif edit == "trace":
                ops.append(_trace_op(rng, m))
            elif edit == "mode":
                if family == "ts":
                    ts_on = not ts_on
                    ops.append({"op": "mode", "ts": ts_on})
                else:
                    ops.append({"op": "mode", "pipe": int(rng.choice([1, 2, 3, 4, 8]))})
            else:
                checkpoints.append(m.s.copy())
                ops.append({"op": "checkpoint", "state": m.s.copy()})
        ops.append(_render_op(rng, m, family, ts_on))
        extra = str(rng.choice(["none", "none", "release", "set_voice", "trace", "mode"]))
        if extra == "release":
            ops.append(_release_op(rng, m, recent))
        elif extra == "set_voice":
            ops.append(_set_voice_op(rng, m, pool, fk, late, recent))
        elif extra == "trace":
            ops.append(_trace_op(rng, m))
        elif extra == "mode" and family == "pipe":
            ops.append({"op": "mode", "pipe": int(rng.choice([1, 2, 3, 4, 8]))})
        elif extra == "mode":
            ts_on = not ts_on
            ops.append({"op": "mode", "ts": ts_on})
    if family == "ts" and not ts_on:
        ts_on = True
        ops.append({"op": "mode", "ts": True})
    ops.append(_render_op(rng, m, family, ts_on))
    ops.append({"op": "checkpoint", "state": m.s.copy()})
    return v, ops


def run_batch_script(v, fk, ops, with_modes):
    """Runs `ops` on a GPU bank: renders back to back, async mixes into two pinned buffers in flight, batches through
    set_voices.  with_modes=False leaves the mode changes out.  Returns one dict per op (test_gpu_edits.check_run)."""
    V = v.shape[0]
    stream = torch.cuda.current_stream()
    nan = float("nan")
    bufs = {}
    for k, op in enumerate(ops):
        if op["op"] not in RENDERS:
            continue
        fr = op["frames"]
        stride = ((fr + 3) & ~3) + 8
        rows = torch.full((V, stride), nan, device="cuda") if op["rows"] or op["op"] == "trace" else None
        bus = None
        if op["op"] == "render" and op["bus"]:
            bus = torch.full((fr + 8,), nan, device="cuda")
        elif op["op"] == "host":
            bus = np.full(fr + 8, np.nan, dtype=np.float32)
        bufs[k] = (rows, bus)
    n_pinned = max([op["frames"] for op in ops if op["op"] == "async"] + [1])
    pinned = [torch.empty(n_pinned, dtype=torch.float32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    in_flight = [None, None]
    res = [{} for _ in ops]

    def collect(slot):
        j = in_flight[slot]
        if j is not None:
            done[slot].synchronize()
            res[j]["bus"] = pinned[slot][:ops[j]["frames"]].numpy().copy()
            in_flight[slot] = None

    torch.cuda.synchronize()
    n_async = 0
    with s2.VoiceBank(v, SR, fk, stream=stream) as bank:
        for k, op in enumerate(ops):
            name = op["op"]
            if name == "mode":
                if with_modes and "pipe" in op:
                    bank.set_pipeline(op["pipe"])
                elif with_modes:
                    bank.set_time_split(op["ts"])
            elif name in RENDERS:
                fr = op["frames"]
                rows, bus = bufs[k]
                stride = 0 if rows is None else rows.stride(0)
                ts0 = bank.time_split_blocks
                if name == "render":
                    bank.render(fr, rows, stride, None if bus is None else bus[4:4 + fr])
                elif name == "host":
                    bank.render_bus_host(fr, rows, stride, out=bus[4:4 + fr])
                elif name == "async":
                    slot = n_async & 1
                    n_async += 1
                    collect(slot)
                    pinned[slot].fill_(nan)
                    bank.render_bus_host_async(fr, pinned[slot], rows, stride)
                    done[slot].record(stream)
                    in_flight[slot] = k
                else:
                    bank.trace_phase(fr, rows, stride)
                res[k]["ts"] = bank.time_split_blocks - ts0
            elif name == "set_voices":
                bank.set_voices(op["idx"], op["descs"])
            elif name == "set_voice":
                for i, d in op["calls"]:
                    bank.set_voice(i, d)
            elif name == "release":
                for i in op["idx"]:
                    bank.release_voice(i)
            elif name == "table":
                bank.set_releases(op["table"])
            elif name == "set_state":
                bank.set_state(op["state"])
            elif name == "checkpoint":
                res[k]["state"] = bank.get_state()
        collect(0)
        collect(1)
        bank.sync()
    torch.cuda.synchronize()
    for k, (rows, bus) in bufs.items():
        fr = ops[k]["frames"]
        if rows is not None:
            assert bool(torch.isnan(rows[:, fr:]).all()), f"{describe(k, ops[k])}: row written past frames"
            res[k]["rows"] = rows[:, :fr].cpu().numpy()
        if bus is not None:
            b = bus if isinstance(bus, np.ndarray) else bus.cpu().numpy()
            assert np.all(np.isnan(b[:4])) and np.all(np.isnan(b[4 + fr:])), f"{describe(k, ops[k])}: bus outside"
            res[k]["bus"] = b[4:4 + fr].copy()
    return res


ORDER_PIPE = [(7, 0), (33, 1), (333, 0), (333, 1), (1000, 0), (1000, 1), (4096, 1)]
ORDER_TS = [(7, 1), (32, 0), (333, 0), (1000, 1)]
ORDER = [(200 + i, V, fk, "pipe") for i, (V, fk) in enumerate(ORDER_PIPE)] + \
        [(300 + i, V, fk, "ts") for i, (V, fk) in enumerate(ORDER_TS)]


@pytest.mark.parametrize("seed,V,fk,family", ORDER, ids=[f"{f}-{V}v-filter{fk}-seed{s}" for s, V, fk, f in ORDER])
def test_batch_call_order(seed, V, fk, family):
    v, ops = make_batch_script(seed, V, fk, family)
    base = run_batch_script(v, fk, ops, with_modes=False)
    check_run(v, fk, ops, base, family, one_stream=True)
    got = run_batch_script(v, fk, ops, with_modes=True)
    check_run(v, fk, ops, got, family, one_stream=False)
    compare_runs(ops, base, got, family)
    if family == "ts":
        # the pitch-modulated voice takes the following block off the time-split path
        k = next(i for i, op in enumerate(ops) if op.get("form") == "pitchmod")
        nxt = next(op for op in ops[k:] if op["op"] in RENDERS)
        assert nxt["ts"] == 0


def test_batch_scripts_cover_the_hazards():
    """Every script stages tables around batches in every named order and batches with every form."""
    for seed, V, fk, family in ORDER:
        _, ops = make_batch_script(seed, V, fk, family)
        joined = " ".join(op["op"] for op in ops)
        for pat in ("table set_voices", "table set_voices table", "set_voices table", "set_voices set_voices"):
            assert pat in joined, (seed, pat)
        forms = {op.get("form") for op in ops if op["op"] == "set_voices"}
        assert {"spread", "all", "one", "pitchmod"} <= forms


# ------------------------------------------------------------------------------ 3. re-patch the whole bank

@pytest.mark.parametrize("V,n_sub", [(1000, 1), (1000, 4), (65536, 1), (65536, 4)])
def test_repatch_whole_bank(V, n_sub):
    """set_voices over every voice in reverse order gives the rows a new bank made from those descriptions renders.
    Pipelined, the batches grow the staging buffers while renders are in flight."""
    fk, T = s2.FILTER_BIQUAD_LP, 2048
    v = _bank(V, fk, 11)
    w = _bank(V, fk, 12)
    rng = np.random.default_rng(3)
    rows = [torch.full((V, T), float("nan"), device="cuda") for _ in range(4)]
    torch.cuda.synchronize()
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        bank.render(T, rows[0], T)
        small = rng.integers(0, V, 5).astype(np.uint32)
        bank.set_voices(small, w[small])
        bank.render(T, rows[1], T)
        order = np.arange(V, dtype=np.uint32)[::-1].copy()
        bank.set_voices(order, w[order])                     # grows both staging buffers
        bank.render(T, rows[2], T)
        bank.sync()
        st = bank.get_state()
    with s2.VoiceBank(w, SR, fk) as fresh:
        fresh.set_pipeline(n_sub)
        fresh.render(T, rows[3], T)
        fresh.sync()
        want_st = fresh.get_state()
    torch.cuda.synchronize()
    assert bool(torch.isfinite(rows[3]).all())
    assert torch.equal(rows[2].view(torch.int32), rows[3].view(torch.int32)), "rows differ from a new bank"
    assert st.tobytes() == want_st.tobytes()


# ------------------------------------------------------------------------------ 4. validation

@pytest.mark.parametrize("n_sub", [1, 4])
def test_invalid_entries_change_nothing(n_sub):
    V, fk, T = 1000, s2.FILTER_BIQUAD_LP, 1024
    v = _bank(V, fk, 21)
    good = _bank(V, fk, 22)
    idx = np.arange(0, V, 97, dtype=np.uint32)
    n = idx.size
    cases = []
    for pos in (0, n // 2, n - 1):
        bad = good[idx].copy()
        bad["pitch_hz"][pos] = float("nan")
        cases.append((idx, bad))
        bad = good[idx].copy()
        bad["damping"][pos] = 0.0                            # second-order filters need damping > 0
        cases.append((idx, bad))
        bad = good[idx].copy()
        bad["osc_kind"][pos] = 7
        cases.append((idx, bad))
        oob = idx.copy()
        oob[pos] = V
        cases.append((oob, good[idx]))
    rows = [torch.full((V, T), float("nan"), device="cuda") for _ in range(2)]
    torch.cuda.synchronize()
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        for ii, dd in cases:
            with pytest.raises(s2.S2Error) as e:
                bank.set_voices(ii, dd)
            assert e.value.code == _lib.S2_ERR_INVALID
        lib = s2.lib()
        assert lib.s2_bank_set_voices(bank._h, n, None, _lib.ptr(good[idx])) == _lib.S2_ERR_INVALID
        assert lib.s2_bank_set_voices(bank._h, n, _lib.ptr(idx), None) == _lib.S2_ERR_INVALID
        assert lib.s2_bank_set_voices(None, n, _lib.ptr(idx), _lib.ptr(good[idx])) == _lib.S2_ERR_INVALID
        assert lib.s2_bank_set_voices(bank._h, 0, None, None) == _lib.S2_OK
        bank.render(T, rows[0], T)
        bank.sync()
    with s2.VoiceBank(v, SR, fk) as untouched:
        untouched.set_pipeline(n_sub)
        untouched.render(T, rows[1], T)
        untouched.sync()
    assert torch.equal(rows[0].view(torch.int32), rows[1].view(torch.int32))


# ------------------------------------------------------------------------------ 5. launch counts

LAUNCH_CASES = [(V, mode) for V in (1, 33, 2048, 65536) for mode in (1, 2, 4, 8, "ts") if not (mode == "ts" and V > 16384)]


@pytest.mark.parametrize("V,mode", LAUNCH_CASES)
def test_set_voices_launches(V, mode):
    """0 for an empty batch; 1 on one stream or time-split; pipelined, one per range with entries (every range for a
    batch of all voices, one for a batch of one voice), with or without a staged table; no gather is added."""
    T = 1024
    voices = bankgen.make_bank(V, 1 << 20)
    table = np.full(V, 3 * T, np.uint32)
    with s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE) as bank:
        if mode == "ts":
            bank.set_time_split(True)
            n_sub = 1
        else:
            bank.set_pipeline(mode)
            n_sub = mode
        every = np.arange(V, dtype=np.uint32)[::-1].copy()
        assert _launches(bank.set_voices, np.zeros(0, np.uint32), voices[:0]) == 0
        for staged in (False, True):
            if staged:
                bank.set_releases(table)
            assert _launches(bank.set_voices, every, voices[every]) == _ranges(V, n_sub)
            assert _launches(bank.set_voices, [V - 1, V - 1], voices[[V - 1, 0]]) == 1
            assert _launches(bank.render, T, None, 0, None) == min(-(-V // 64), n_sub)
        bank.sync()


# ------------------------------------------------------------------------------ 6. no wait

def test_set_voices_does_not_wait_on_one_stream():
    V = 4096
    voices = bankgen.make_bank(V, 1 << 20)
    stream = torch.cuda.current_stream()
    idx = np.arange(0, V, 7, dtype=np.uint32)
    with s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE, stream=stream) as bank:
        bank.set_voices(idx, voices[idx])                    # the staging buffers exist from here on
        bank.sync()
        done = torch.cuda.Event()
        torch.cuda._sleep(2_000_000_000)                     # about a second of spinning on the bank's stream
        done.record(stream)
        bank.set_voices(idx, voices[idx])
        assert not done.query(), "set_voices waited for the bank's stream"
        bank.sync()


def test_set_voices_does_not_wait_behind_pipelined_renders():
    V = 65536
    voices = bankgen.make_bank(V, 1 << 22, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    stream = torch.cuda.current_stream()
    idx = np.arange(0, V, 101, dtype=np.uint32)
    table = np.full(V, 1 << 21, np.uint32)
    with s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, stream=stream) as bank:
        bank.set_pipeline(4)
        bank.set_voices(idx, voices[idx])
        bank.sync()
        bank.set_releases(table)
        bank.render(1 << 20, None, 0, None)                 # tens of milliseconds on every range
        bank.join(stream)
        done = torch.cuda.Event()
        done.record(stream)
        bank.set_voices(idx, voices[idx])
        bank.set_releases(table)                            # supersedes the table the batch patched
        bank.set_voices(idx[:3], voices[idx[:3]])
        assert not done.query(), "set_voices waited for the pipelined renders"
        bank.sync()
