"""Edits between renders — set_voice, release_voice, set_releases, set_state, mode changes — against the oracle in
every render mode.

Between the calls a streaming caller makes and the kernels sits the bank's host layer (s2_capi.cu): the slot
permutation, host mirrors of the voice descriptions and offsets (they decide time-split blocks and offset overflow),
the pipelined mode's staged note-off table and the ordering of the time-split phase pre-pass.  Seeded scripts of edits
and renders run on a GPU bank and on a host model that applies each edit as the reference does, in call order
(synth.rs:61-80, main.rs:138-147), and advances with the oracle:

    set_voice(i, d)     descs[i] = d; states[i] = fresh state at d's frame offset
    release_voice(i)    descs[i].release_offset = states[i].frame_offset
    set_releases(t)     descs.release_offset = t
    set_state(s)        states = s
    render / trace      advance by the call's frames

Each script runs twice: with its mode changes (pipeline 1-8 or time-split on/off) and without them, on one stream.
Pipelined runs must give the same bytes as the one-stream run (rows, bus, phase traces, state); time-split runs the
same within the north-star tolerance, with exactly the time-split blocks the host rule predicts.
"""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
import synth2_b200 as s2  # noqa: E402
from busref import U, assert_bus_within_bound, reference_order_bus  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402
from test_gpu_parity import TOL_ABS, assert_parity  # noqa: E402

pytestmark = pytest.mark.gpu

SR = 48000
RENDERS = ("render", "host", "async", "trace")
FRAMES = (17, 100, 1000, 3001, 64, 1024, 2048, 4096)
FRAMES_TS = (1024, 2048, 4096, 4096, 1024, 1000, 17, 3001)      # mostly whole 1,024-frame blocks
TS_LIMIT = 1 << 24                                               # time-split blocks keep offsets below 2^24
ALL_KINDS = (s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_TRIANGLE, s2.OSC_SINE)


def _sweep(fk):
    return bankgen.MOD_TO_LPF_ONE_POLE if fk == s2.FILTER_ONE_POLE else bankgen.MOD_TO_LPF_BIQUAD


def _bank(V, fk, seed, late=False):
    """V voices for filter `fk`: all kinds (or no sine, on odd seeds), some noise, cutoff followers and resting
    cutoffs, a mod envelope with a sustain and a release (so a note-off moves a follower's cutoff), started at
    random offsets (late: past the 200 ms mod decay, so most cutoffs rest), 30 % held, some inactive."""
    rng = np.random.default_rng(seed)
    kinds = ALL_KINDS if seed % 2 == 0 else ALL_KINDS[:3]
    v = bankgen.make_bank(V, 16384, first_voice=seed * 4099, kinds=kinds, mod_to_lpf_choices=_sweep(fk))
    v["osc_kind"] = rng.choice(kinds, V)
    v["noise_amt"] = rng.choice([0.0, 0.0, 0.25], V)
    v["mod_sustain"] = rng.choice([0.0, 0.5], V)
    v["mod_release_ms"] = rng.choice([0.0, 40.0], V)
    if fk == s2.FILTER_BIQUAD_BP:
        v["damping"] += 2.0          # the field is the quality factor here; theta / (2 Q) must stay below pi / 4
    start = 10000 if late else 0
    v["frame_offset"] = np.where(rng.random(V) < 0.6, start + rng.integers(0, 30000, V), start)
    rel = v["frame_offset"].astype(np.int64) + rng.integers(-2000, 20000, V)
    v["release_offset"] = np.where(rng.random(V) < 0.3, s2.NO_RELEASE, np.maximum(rel, 0))
    v["active"] = rng.random(V) < 0.85
    v["active"][V // 2] = 0
    v["active"][0] = 1
    return v


class _Model:
    """The reference bank as its caller sees it: descriptions and carried states, advanced by the oracle."""

    def __init__(self, v, fk):
        self.d = v.copy()
        self.s = oracle.bank_init_states(v)
        self.fk = fk

    def render(self, frames, rows=True):
        out, _ = oracle.bank_render(self.d, self.s, SR, self.fk, frames, want_voices=rows, want_bus=False, nthreads=8)
        return out

    def set_voice(self, i, desc):
        self.d[i] = desc[0]
        self.s[i] = oracle.bank_init_states(desc)[0]

    def release_voice(self, i):
        self.d["release_offset"][i] = self.s["frame_offset"][i]

    def set_releases(self, table):
        self.d["release_offset"] = table

    def set_state(self, state):
        self.s = state.copy()

    def ts_block(self, frames):
        """The host rule of a time-split block (given time-split on and rows requested): whole 1,024-frame blocks,
        every active voice without pitch modulation and below 2^24 at the block's end."""
        act = self.d["active"] != 0
        return (frames % 1024 == 0 and not np.any(self.d["mod_env_to_osc_freq"][act] != 0.0)
                and bool(np.all(self.s["frame_offset"][act].astype(np.int64) + frames <= TS_LIMIT)))


# ------------------------------------------------------------------------------ scripts

def _fresh(rng, pool, late):
    d = pool[int(rng.integers(pool.shape[0]))][None].copy()
    d["active"] = 1
    off = int(rng.integers(12000, 40000)) if late and rng.random() < 0.7 else int(rng.choice([0, rng.integers(0, 20000)]))
    d["frame_offset"] = off
    d["release_offset"] = s2.NO_RELEASE if rng.random() < 0.5 else off + int(rng.integers(0, 8000))
    return d


def _set_voice_op(rng, m, pool, fk, late, recent):
    """One to three set_voice calls of one form: retrigger an active voice, fill an inactive slot, deactivate a
    voice, change the oscillator kind (to or from sine), or turn a cutoff follower into a resting voice or back."""
    V = m.d.shape[0]
    form = str(rng.choice(["retrigger", "fill", "deactivate", "kind", "follower"]))
    active = np.flatnonzero(m.d["active"] != 0)
    inactive = np.flatnonzero(m.d["active"] == 0)
    cand = inactive if form == "fill" else active
    if cand.size == 0:
        cand = np.arange(V)
    idx = rng.choice(cand, size=min(int(rng.integers(1, 4)), cand.size), replace=False)
    calls = []
    for i in map(int, idx):
        if form in ("retrigger", "fill"):
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
        calls.append((i, d))
        recent.append(i)
    return {"op": "set_voice", "form": form, "calls": calls}


def _release_op(rng, m, recent):
    """release_voice on a held active voice, an already released one, an inactive one and a recently set one."""
    act = m.d["active"] != 0
    released = m.d["release_offset"].astype(np.int64) <= m.s["frame_offset"].astype(np.int64)
    idx = []
    for group in (np.flatnonzero(act & ~released), np.flatnonzero(act & released), np.flatnonzero(~act),
                  np.asarray(recent[-4:], dtype=np.int64)):
        if group.size and rng.random() < 0.75:
            i = int(rng.choice(group))
            if i not in idx:
                idx.append(i)
    if not idx:
        idx = [int(rng.integers(m.d.shape[0]))]
    for i in idx:
        m.release_voice(i)
    return {"op": "release", "idx": idx}


def _table_op(rng, m):
    """A note-off table: 40 % of the voices get NO_RELEASE, a past, the current or a future offset."""
    V = m.d.shape[0]
    off = m.s["frame_offset"].astype(np.int64)
    t = m.d["release_offset"].astype(np.int64)
    pick = rng.random(V) < 0.4
    what = rng.integers(0, 4, V)
    new = np.select([what == 0, what == 1, what == 2],
                    [s2.NO_RELEASE, np.maximum(off - rng.integers(1, 5000, V), 0), off],
                    off + rng.integers(1, 6000, V))
    t = np.where(pick, new, t)
    t = np.clip(t, 0, 0xFFFFFFFF).astype(np.uint32)
    m.set_releases(t)
    return {"op": "table", "table": t}


def _synthetic_state(rng, m):
    """A state no render made: half the voices get a random phase with has_phase 0 or 1, non-zero filter state and
    an offset moved forward; a few sit just below 2^24."""
    V = m.d.shape[0]
    s = m.s.copy()
    sel = rng.random(V) < 0.5
    n = int(sel.sum())
    s["has_phase"][sel] = rng.integers(0, 2, n)
    s["phase"][sel] = rng.random(n).astype(np.float32)
    s["lpf_last"][sel] = rng.uniform(-0.5, 0.5, n)
    for k, a in (("x1", 1.0), ("x2", 1.0), ("y1", 0.5), ("y2", 0.5)):
        s[k][sel] = rng.uniform(-a, a, n)
    s["frame_offset"][sel] += rng.integers(0, 40000, n).astype(np.uint32)
    near = rng.random(V) < 0.1
    s["frame_offset"][near] = TS_LIMIT - rng.integers(0, 6000, int(near.sum()))
    m.set_state(s)
    return {"op": "set_state", "state": s.copy(), "how": "synthetic"}


def make_script(seed, V, fk, family):
    """(voices, ops) of one seeded script; every op carries what the model expects of it."""
    rng = np.random.default_rng(seed)
    late = family == "ts"
    v = _bank(V, fk, seed, late=late)
    pool = _bank(64, fk, 50000 + seed, late=late)
    m = _Model(v, fk)
    ts_on = family == "ts"
    ops = [{"op": "mode", "ts": True} if ts_on else {"op": "mode", "pipe": int(rng.choice([2, 3, 4, 8]))}]
    checkpoints, recent = [], []
    n_ops = int(rng.integers(8, 16))
    frames_pool = FRAMES_TS if family == "ts" else FRAMES
    while len(ops) < n_ops:
        last = len(ops) == n_ops - 1
        prev = ops[-1]["op"]
        if last or (prev not in RENDERS and rng.random() < 0.6) or rng.random() < 0.25:
            call = str(rng.choice(["render", "render", "host", "async", "trace"]))
            fr = int(rng.choice(frames_pool))
            op = {"op": call, "frames": fr}
            if call == "render":
                op["rows"], op["bus"] = [(True, False), (False, True), (True, True), (True, True)][int(rng.integers(4))]
            elif call in ("host", "async"):
                op["rows"], op["bus"] = bool(rng.random() < 0.75), True
            else:
                op["rows"], op["bus"] = False, False
            op["ts"] = int(ts_on and call != "trace" and op["rows"] and m.ts_block(fr))
            op["expect"] = m.render(fr)
            ops.append(op)
            continue
        what = str(rng.choice(["set_voice", "set_voice", "release", "table", "state", "mode"]))
        if prev == "table" and family == "pipe" and rng.random() < 0.5:
            what = "mode"                       # a pipeline change with a table staged
        if what == "set_voice":
            ops.append(_set_voice_op(rng, m, pool, fk, late, recent))
        elif what == "release":
            ops.append(_release_op(rng, m, recent))
        elif what == "table":
            ops.append(_table_op(rng, m))
        elif what == "mode":
            if family == "ts":
                ts_on = not ts_on
                ops.append({"op": "mode", "ts": ts_on})
            else:
                ops.append({"op": "mode", "pipe": int(rng.choice([1, 2, 3, 4, 8]))})
        elif checkpoints and rng.random() < 0.5:
            s = checkpoints[int(rng.integers(len(checkpoints)))]
            m.set_state(s)
            ops.append({"op": "set_state", "state": s.copy(), "how": "checkpoint"})
        elif rng.random() < 0.5:
            ops.append(_synthetic_state(rng, m))
        else:
            checkpoints.append(m.s.copy())
            ops.append({"op": "checkpoint", "state": m.s.copy()})
    ops.append({"op": "checkpoint", "state": m.s.copy()})
    return v, ops


def describe(k, op):
    extra = {"mode": lambda: f"pipe {op['pipe']}" if "pipe" in op else f"time-split {op['ts']}",
             "set_voice": lambda: f"{op['form']} {[i for i, _ in op['calls']]}",
             "release": lambda: str(op["idx"]),
             "set_state": lambda: op["how"]}.get(op["op"], lambda: "")
    if op["op"] in RENDERS:
        return f"op {k} {op['op']} {op['frames']} frames rows={op['rows']} bus={op['bus']}"
    return f"op {k} {op['op']} {extra()}"


# ------------------------------------------------------------------------------ running a script on the GPU

def run_script(v, fk, ops, with_modes):
    """Runs `ops` on a GPU bank, renders back to back (the bank drains itself where an edit needs it), async mixes
    into two pinned buffers in flight.  with_modes=False leaves the mode changes out.  Returns one dict per op."""
    V = v.shape[0]
    stream = torch.cuda.current_stream()
    nan = float("nan")
    bufs = {}
    for k, op in enumerate(ops):
        if op["op"] not in RENDERS:
            continue
        fr = op["frames"]
        stride = ((fr + 3) & ~3) + 8                       # padded: nothing may land between frames and stride
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

    torch.cuda.synchronize()                 # the NaN fills are done before any of the bank's streams writes
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


# ------------------------------------------------------------------------------ checks

STATE_KEYS = {s2.FILTER_ONE_POLE: ("lpf_last",), s2.FILTER_BIQUAD_LP: ("x1", "x2", "y1", "y2"),
              s2.FILTER_BIQUAD_HP: ("x1", "x2", "y1", "y2"), s2.FILTER_BIQUAD_BP: ("x1", "x2", "y1", "y2"),
              s2.FILTER_FIRST_ORDER_LP: ("x1", "y1"), s2.FILTER_FIRST_ORDER_HP: ("x1", "y1")}


def check_state(got, want, fk, what):
    """Phase, has_phase and offsets bit-exact; the filter's own state within the parity tolerance."""
    assert np.array_equal(got["frame_offset"], want["frame_offset"]), f"{what}: frame offsets"
    assert np.array_equal(got["has_phase"], want["has_phase"]), f"{what}: has_phase"
    bad = np.flatnonzero(got["phase"].view(np.uint32) != want["phase"].view(np.uint32))
    assert bad.size == 0, f"{what}: phase differs for voices {bad[:8]}"
    for key in STATE_KEYS[fk]:
        np.testing.assert_allclose(got[key], want[key], atol=TOL_ABS * 4, rtol=0, err_msg=f"{what}: {key}")


def check_bus(bus, rows, V, path, what):
    """A bus against the rows of the same call: the reference's sequential voice-order sum, byte for byte, up to 32
    voices; the summation tree's error bound above."""
    if V <= 32:
        want = reference_order_bus(rows)
        assert bus.tobytes() == want.tobytes(), (
            f"{what}: bus differs from the voice-order sum at {int(np.sum(bus.view(np.uint32) != want.view(np.uint32)))}"
            f" of {bus.size} frames")
    else:
        assert_bus_within_bound(bus, rows, V, path, what)


def check_bus_near_reference(bus, ref_rows, what):
    """A bus of a call without rows, against the oracle's rows: each row may be off by the parity tolerance."""
    exact = ref_rows.astype(np.float64).sum(axis=0)
    mag = np.abs(ref_rows.astype(np.float64)).sum(axis=0)
    sounding = int(np.count_nonzero(np.any(ref_rows != 0.0, axis=1)))
    tol = TOL_ABS * max(1.0, float(np.max(np.abs(ref_rows)))) * sounding + 64 * U * mag
    err = np.abs(bus.astype(np.float64) - exact)
    assert np.all(np.isfinite(bus)) and np.all(err <= tol), f"{what}: bus off the oracle's sum by {err.max():.3e}"


def check_run(v, fk, ops, res, family, one_stream):
    """One run against the model's expectations; `one_stream`: this run left the mode changes out."""
    V = v.shape[0]
    for k, op in enumerate(ops):
        what = f"{'one-stream' if one_stream else family} run, {describe(k, op)}"
        r = res[k]
        if op["op"] in RENDERS:
            want_ts = 0 if one_stream else op["ts"]
            assert r["ts"] == want_ts, f"{what}: {r['ts']} time-split blocks, the host rule says {want_ts}"
            if op["op"] == "trace":
                assert np.all(np.isfinite(r["rows"])), what
                continue
            if op["rows"]:
                assert_parity(op["expect"], r["rows"], what)
                if op["bus"]:
                    check_bus(r["bus"], r["rows"], V, "time_split" if r["ts"] else "default", what)
            elif op["bus"]:
                check_bus_near_reference(r["bus"], op["expect"], what)
        elif op["op"] == "checkpoint":
            check_state(r["state"], op["state"], fk, what)


def compare_runs(ops, base, got, family):
    """The run with mode changes against the one-stream run: pipelined byte for byte, time-split within tolerance
    (phase traces, phases and offsets still byte for byte)."""
    for k, op in enumerate(ops):
        what = f"{family} run against one-stream, {describe(k, op)}"
        for key in ("rows", "bus", "state"):
            if key not in base[k]:
                continue
            a, b = base[k][key], got[k][key]
            if family == "pipe" or op["op"] == "trace":
                assert a.tobytes() == b.tobytes(), f"{what}: {key} differs"
            elif key == "state":
                for field in ("phase", "has_phase", "frame_offset"):
                    assert a[field].tobytes() == b[field].tobytes(), f"{what}: {field} differs"
            else:
                assert_parity(a, b, f"{what}: {key}")


PIPE_CASES = [(7, 0), (7, 3), (32, 1), (32, 5), (33, 2), (33, 4), (333, 0), (333, 1), (333, 3), (640, 2), (640, 5),
              (640, 1), (1000, 0), (1000, 1), (1000, 4), (1000, 3)]
TS_CASES = [(7, 0), (32, 1), (32, 0), (33, 1), (333, 0), (640, 1), (1000, 0), (1000, 1)]
SCRIPTS = [(i, V, fk, "pipe") for i, (V, fk) in enumerate(PIPE_CASES)] + \
          [(100 + i, V, fk, "ts") for i, (V, fk) in enumerate(TS_CASES)]


@pytest.mark.parametrize("seed,V,fk,family", SCRIPTS, ids=[f"{f}-{V}v-filter{fk}-seed{s}" for s, V, fk, f in SCRIPTS])
def test_edit_script(seed, V, fk, family):
    """A seeded script of renders (rows, bus or both; host copies; async copies; phase traces) and edits (every form
    of set_voice, release_voice, note-off tables, checkpoints and synthetic states, mode changes) against the model
    after every call, and against the same script on one stream."""
    v, ops = make_script(seed, V, fk, family)
    base = run_script(v, fk, ops, with_modes=False)
    check_run(v, fk, ops, base, family, one_stream=True)
    got = run_script(v, fk, ops, with_modes=True)
    check_run(v, fk, ops, got, family, one_stream=False)
    compare_runs(ops, base, got, family)


def test_scripts_cover_the_vocabulary():
    """The seeded scripts together use every call, every set_voice form, every release case, tables with all four
    kinds of entry, both kinds of set_state, every pipeline split, time-split toggles and qualifying blocks."""
    seen = set()
    for seed, V, fk, family in SCRIPTS:
        _, ops = make_script(seed, V, fk, family)
        for op in ops:
            seen.add(op["op"])
            if op["op"] == "set_voice":
                seen.add(op["form"])
            elif op["op"] == "set_state":
                seen.add(op["how"])
            elif op["op"] == "mode":
                seen.add(f"pipe{op['pipe']}" if "pipe" in op else f"ts{int(op['ts'])}")
            elif op["op"] in RENDERS and op.get("ts"):
                seen.add("ts-block")
            elif op["op"] in RENDERS and family == "ts" and op["frames"] % 1024:
                seen.add("ts-ragged")
    want = set(RENDERS) | {"set_voice", "release", "table", "checkpoint", "retrigger", "fill", "deactivate", "kind",
                           "follower", "synthetic", "pipe1", "pipe2", "pipe3", "pipe4", "pipe8", "ts0", "ts1",
                           "ts-block", "ts-ragged"}
    assert want <= seen, sorted(want - seen)


# ------------------------------------------------------------------------------ named regressions

def _staged_table_case(n_sub, edit):
    """Render, stage a note-off table, edit some voices, render: (rows of both renders, final state) on the GPU and
    in the model.  edit = "set_voice": the table gives the voices a past offset, then fresh held notes replace them;
    edit = "release": the table holds them (NO_RELEASE), then release_voice releases them."""
    V, fk = 1000, s2.FILTER_BIQUAD_LP
    v = _bank(V, fk, 7)
    v["active"] = 1
    v["release_offset"] = s2.NO_RELEASE
    picked = np.arange(3, V, 97)
    m = _Model(v, fk)
    want = [m.render(2048)]
    off = m.s["frame_offset"].astype(np.int64)
    table = (off + 4000).astype(np.uint32)
    table[picked] = (off[picked] - 100) if edit == "set_voice" else s2.NO_RELEASE   # set_voice: before the new note
    m.set_releases(table)
    fresh = {}
    for i in picked:
        if edit == "set_voice":
            d = v[i:i + 1].copy()
            d["frame_offset"] = 20000
            d["release_offset"] = s2.NO_RELEASE
            fresh[int(i)] = d
            m.set_voice(int(i), d)
        else:
            m.release_voice(int(i))
    want.append(m.render(4096))
    rows = [torch.full((V, fr), float("nan"), device="cuda") for fr in (2048, 4096)]
    torch.cuda.synchronize()
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        bank.render(2048, rows[0], 2048)
        bank.set_releases(table)
        for i in picked:
            if edit == "set_voice":
                bank.set_voice(int(i), fresh[int(i)])
            else:
                bank.release_voice(int(i))
        bank.render(4096, rows[1], 4096)
        bank.sync()
        st = bank.get_state()
    return [r.cpu().numpy() for r in rows], st, want, m.s, picked


@pytest.mark.parametrize("n_sub", [1, 2, 4, 8])
def test_set_voice_after_a_staged_note_off_table(n_sub):
    """set_releases(t), then set_voice(i, fresh held note), then render: the later note-on wins (the reference
    applies events in arrival order), so voice i does not start released at t[i], an offset in its past."""
    got, st, want, want_st, picked = _staged_table_case(n_sub, "set_voice")
    for k in range(2):
        assert_parity(want[k][picked], got[k][picked], f"pipeline {n_sub}, render {k}: the fresh notes")
        assert_parity(want[k], got[k], f"pipeline {n_sub}, render {k}")
    check_state(st, want_st, s2.FILTER_BIQUAD_LP, f"pipeline {n_sub}")
    if n_sub > 1:
        base, base_st, _, _, _ = _staged_table_case(1, "set_voice")
        assert all(a.tobytes() == b.tobytes() for a, b in zip(base, got)) and base_st.tobytes() == st.tobytes()


@pytest.mark.parametrize("n_sub", [1, 2, 4, 8])
def test_release_voice_after_a_staged_note_off_table(n_sub):
    """set_releases(t) with t[i] = NO_RELEASE, then release_voice(i): voice i releases at its current offset."""
    got, st, want, want_st, picked = _staged_table_case(n_sub, "release")
    for k in range(2):
        assert_parity(want[k][picked], got[k][picked], f"pipeline {n_sub}, render {k}: the released voices")
        assert_parity(want[k], got[k], f"pipeline {n_sub}, render {k}")
    check_state(st, want_st, s2.FILTER_BIQUAD_LP, f"pipeline {n_sub}")
    if n_sub > 1:
        base, base_st, _, _, _ = _staged_table_case(1, "release")
        assert all(a.tobytes() == b.tobytes() for a, b in zip(base, got)) and base_st.tobytes() == st.tobytes()


def _trace_then_renders(n_sub, staged):
    """trace_phase(8,192) on a 16,384-voice bank, then 8 renders with rows and a bus, no host sync in between,
    joined at the end.  staged: a note-off table set just before the trace, releasing voices inside the traced
    frames; a third of the voices follow the mod envelope with their pitch, so the release shows in the trace."""
    V, T, N, fk = 16384, 2048, 8, s2.FILTER_ONE_POLE
    v = bankgen.make_bank(V, 8192 + N * T, kinds=ALL_KINDS)
    v["release_offset"] = s2.NO_RELEASE
    v["mod_sustain"] = 0.5
    v["mod_release_ms"] = 30.0
    v["mod_env_to_osc_freq"][::3] = 0.5
    rng = np.random.default_rng(5)
    table = np.where(rng.random(V) < 0.5, rng.integers(0, 8192, V), s2.NO_RELEASE).astype(np.uint32)
    phase = torch.full((V, 8192), float("nan"), device="cuda")
    rows = [torch.full((V, T), float("nan"), device="cuda") for _ in range(N)]
    buses = [torch.full((T,), float("nan"), device="cuda") for _ in range(N)]
    torch.cuda.synchronize()
    with s2.VoiceBank(v, SR, fk) as bank:
        bank.set_pipeline(n_sub)
        if staged:
            bank.set_releases(table)
        bank.trace_phase(8192, phase)
        for i in range(N):
            bank.render(T, rows[i], T, buses[i])
        bank.join(None)
        torch.cuda.synchronize()
        st = bank.get_state()
    return (phase.cpu().numpy(), torch.cat(rows, dim=1).cpu().numpy(), torch.cat(buses).cpu().numpy(), st)


@pytest.mark.parametrize("staged", [False, True], ids=["no-table", "staged-table"])
def test_trace_is_ordered_before_pipelined_renders(staged):
    """A phase trace on a pipelined bank, then renders without a sync: trace, rows, bus and final state equal the
    same calls on a one-stream bank byte for byte.  With a staged table the trace render applies it."""
    want = _trace_then_renders(1, staged)
    got = _trace_then_renders(4, staged)
    assert all(np.all(np.isfinite(a)) for a in want[:3])
    for name, a, b in zip(("phase trace", "rows", "bus", "state"), want, got):
        assert a.tobytes() == b.tobytes(), f"{name} differs from the one-stream bank"
