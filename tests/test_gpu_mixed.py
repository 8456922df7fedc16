"""Mixed-filter voice banks (s2_bank_create_mixed): a filter kind per voice, every kind rendered by one launch.

A voice's output bits do not depend on its warp-mates (test_paths_agree_bitwise, test_lane_pair_layouts_agree_bitwise),
so a mixed bank is checked bit for bit against the single-kind banks built from the same voices: a twin of K banks
(one per kind present) receives the same calls, with voice indices mapped into each bank, and must produce the same
rows, meters, phase traces and carried state.  The bus is checked against the voice-order sum (up to 32 voices) or the
summation-tree bound (wider banks), and across render modes bit for bit.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import synth2_b200 as s2  # noqa: E402
from busref import U, assert_bus_within_bound, reference_order_bus  # noqa: E402
from synth2_b200 import _lib, bankgen  # noqa: E402
from test_gpu_edits import SR, _bank  # noqa: E402
from test_gpu_parity import assert_parity, oracle_bank_render  # noqa: E402

pytestmark = pytest.mark.gpu

KINDS = (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP, s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP,
         s2.FILTER_FIRST_ORDER_LP, s2.FILTER_FIRST_ORDER_HP)
FRAMES = (17, 1000, 64, 2051)              # x16 blocks and `frames % 16` tails, ragged and whole tiles
WIDTHS = (1, 7, 32, 33, 333, 1000, 65536)


def mixed_voices(V, seed, n_kinds=6):
    """V voices with random filter kinds (at least two where V allows): each voice is drawn from test_gpu_edits's
    bank for its own kind (all oscillator kinds, noise, cutoff followers and resting cutoffs, inactive voices), and
    a tenth of them also modulate their pitch."""
    rng = np.random.default_rng(seed)
    kinds = rng.choice(KINDS[:n_kinds], V).astype(np.uint32)
    if V > 1 and n_kinds > 1 and np.all(kinds == kinds[0]):
        kinds[-1] = KINDS[(KINDS.index(int(kinds[0])) + 1) % n_kinds]
    v = np.zeros(V, dtype=s2.VOICE_DESC)
    for k in np.unique(kinds):
        sel = kinds == k
        v[sel] = _bank(V, int(k), seed)[sel]
    v["mod_env_to_osc_freq"] = np.where(rng.random(V) < 0.1, rng.choice([-0.5, 0.25], V), 0.0)
    return v, kinds


def n_slots(kinds):
    """Slots of a mixed bank: each kind group but the last padded to whole warps of 32."""
    sizes = [int(np.sum(kinds == k)) for k in KINDS if np.any(kinds == k)]
    return sum(-(-n // 32) * 32 for n in sizes[:-1]) + sizes[-1]


def _meters(V):
    return (torch.zeros(V, device="cuda", dtype=torch.float64), torch.zeros(V, device="cuda", dtype=torch.float32))


def _stride(fr):
    return (fr + 3) & ~3


class Twin:
    """The single-kind banks of a mixed bank's voices, driven as one bank: voice i of the mixed bank is voice
    local[i] of banks[kinds[i]]."""

    def __init__(self, voices, kinds):
        self.kinds = kinds
        self.V = voices.shape[0]
        self.members = {int(k): np.flatnonzero(kinds == k) for k in np.unique(kinds)}
        self.local = np.zeros(self.V, dtype=np.int64)
        for m in self.members.values():
            self.local[m] = np.arange(m.size)
        self.banks = {k: s2.VoiceBank(voices[m], SR, k) for k, m in self.members.items()}
        self.meters = {k: _meters(m.size) for k, m in self.members.items()}

    def close(self):
        for b in self.banks.values():
            b.close()

    def set_pipeline(self, n):
        for b in self.banks.values():
            b.set_pipeline(n)

    def render(self, fr, metered=True):
        rows = torch.empty((self.V, fr), device="cuda")
        for k, m in self.members.items():
            out = torch.full((m.size, _stride(fr)), float("nan"), device="cuda")
            self.banks[k].render(fr, out, _stride(fr), None, *(self.meters[k] if metered else (None, None)))
            self.banks[k].sync()
            rows[torch.from_numpy(m).cuda()] = out[:, :fr]
        return rows

    def trace(self, fr):
        ph = torch.empty((self.V, fr), device="cuda")
        for k, m in self.members.items():
            out = torch.full((m.size, fr), float("nan"), device="cuda")
            self.banks[k].trace_phase(fr, out, fr)
            ph[torch.from_numpy(m).cuda()] = out
        return ph

    def set_voice(self, i, d):
        self.banks[int(self.kinds[i])].set_voice(int(self.local[i]), d)

    def set_voices(self, idx, ds):
        for k, m in self.members.items():
            sel = self.kinds[idx] == k
            if np.any(sel):
                self.banks[k].set_voices(self.local[idx[sel]], ds[sel])

    def release_voice(self, i):
        self.banks[int(self.kinds[i])].release_voice(int(self.local[i]))

    def set_releases(self, table):
        for k, m in self.members.items():
            self.banks[k].set_releases(np.ascontiguousarray(table[m]))

    def get_state(self):
        st = np.zeros(self.V, dtype=s2.VOICE_STATE)
        for k, m in self.members.items():
            st[m] = self.banks[k].get_state()
        return st

    def set_state(self, st):
        for k, m in self.members.items():
            self.banks[k].set_state(np.ascontiguousarray(st[m]))

    def meter_values(self):
        s, p = np.zeros(self.V), np.zeros(self.V, dtype=np.float32)
        for k, m in self.members.items():
            s[m] = self.meters[k][0].cpu().numpy()
            p[m] = self.meters[k][1].cpu().numpy()
        return s, p


def render_mixed(bank, fr, meters=None, bus=False, canary=False):
    """Rows [V, fr] of one render, and the bus.  canary: the buffer has one more row past the last voice, which must
    keep its value (an off-by-one row index; a padding slot's row, 0xffffffff, would address far outside the buffer
    and fault instead)."""
    V = bank.n_voices
    out = torch.full((V + 1, _stride(fr)), float("nan"), device="cuda")
    out[V] = 7.0
    b = torch.full((fr,), float("nan"), device="cuda") if bus else None
    bank.render(fr, out, _stride(fr), b, *(meters if meters is not None else (None, None)))
    bank.sync()
    if canary:
        assert torch.all(out[V] == 7.0), "a padding slot wrote past the caller's rows"
    return out[:V, :fr], b


def same(a, b, what):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    b = b.cpu().numpy() if hasattr(b, "cpu") else np.asarray(b)
    assert a.shape == b.shape, what
    assert a.tobytes() == b.tobytes(), f"{what}: {np.sum(a.view(np.uint8) != b.view(np.uint8))} bytes differ"


# ------------------------------------------------------------------------------ 1. against single-kind banks

@pytest.mark.parametrize("V", WIDTHS)
def test_rows_meters_state_match_single_kind_banks(V):
    voices, kinds = mixed_voices(V, seed=V)
    frames = FRAMES if V < 65536 else (1000, 2051)
    twin = Twin(voices, kinds)
    meters = _meters(V)
    try:
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
            for fr in frames:
                got, _ = render_mixed(bank, fr, meters, canary=True)
                same(got, twin.render(fr), f"V={V} rows of a {fr}-frame render")
            same(bank.get_state(), twin.get_state(), f"V={V} state")
            s, p = twin.meter_values()
            same(meters[0], s, f"V={V} sum_sq")
            same(meters[1], p, f"V={V} peak")
    finally:
        twin.close()


# ------------------------------------------------------------------------------ 2. one kind = s2_bank_create

@pytest.mark.parametrize("fk", KINDS)
@pytest.mark.parametrize("V", (7, 1000))
def test_one_kind_is_bank_create(fk, V):
    voices = _bank(V, fk, seed=fk + V)
    kinds = np.full(V, fk, dtype=np.uint32)
    for n_sub in (1, 4):
        res = []
        for make in (lambda: s2.VoiceBank(voices, SR, fk), lambda: s2.VoiceBank.mixed(voices, kinds, SR)):
            meters = _meters(V)
            with make() as bank:
                bank.set_pipeline(n_sub)
                outs = [render_mixed(bank, fr, meters, bus=True) for fr in FRAMES]
                res.append((outs, bank.get_state(), meters))
        (a, sa, ma), (b, sb, mb) = res
        for (ra, ba), (rb, bb), fr in zip(a, b, FRAMES):
            same(rb, ra, f"rows fk={fk} n_sub={n_sub} {fr}")
            same(bb, ba, f"bus fk={fk} n_sub={n_sub} {fr}")
        same(sb, sa, "state")
        same(mb[0], ma[0], "sum_sq")
        same(mb[1], ma[1], "peak")


# ------------------------------------------------------------------------------ 3. bus

@pytest.mark.parametrize("V", (2, 7, 32))
def test_narrow_bus_adds_in_voice_order(V):
    """Several kinds in up to 32 voices occupy several warps; the bus is still the reference's voice-order sum."""
    voices, kinds = mixed_voices(V, seed=100 + V)
    assert len(np.unique(kinds)) >= 2
    for n_sub in (1, 2, 8):
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank, s2.VoiceBank.mixed(voices, kinds, SR) as no_rows:
            bank.set_pipeline(n_sub)
            no_rows.set_pipeline(n_sub)
            for fr in FRAMES:
                rows, bus = render_mixed(bank, fr, bus=True)
                same(bus, reference_order_bus(rows.cpu().numpy()), f"V={V} n_sub={n_sub} bus of {fr} frames")
                bus2 = torch.full((fr,), float("nan"), device="cuda")
                no_rows.render(fr, None, 0, bus2)
                no_rows.sync()
                same(bus2, bus, f"V={V} n_sub={n_sub} bus without rows, {fr} frames")


@pytest.mark.parametrize("V", (333, 4096))
def test_wide_bus_is_deterministic_and_bounded(V):
    voices, kinds = mixed_voices(V, seed=200 + V)
    buses = {}
    for n_sub in (1, 2, 4, 8):
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
            bank.set_pipeline(n_sub)
            buses[n_sub] = []
            for fr in (1024, 2051, 4096):
                rows, bus = render_mixed(bank, fr, bus=True)
                assert_bus_within_bound(bus, rows, n_slots(kinds), "default", f"V={V} n_sub={n_sub} {fr}")
                buses[n_sub].append(bus.cpu().numpy())
    for n_sub in (2, 4, 8):
        for a, b in zip(buses[1], buses[n_sub]):
            same(b, a, f"V={V} bus n_sub={n_sub} against the default mode")


# ------------------------------------------------------------------------------ 4. pipelined mode with edits

def _edit_script(V, seed, voices, kinds):
    """Renders with a staged note-off table and a set_voices batch between them (each entry keeps its voice's kind:
    drawn from a fresh bank of that kind)."""
    rng = np.random.default_rng(seed)
    ops = []
    for fr in (1000, 2051, 64, 4096, 17):
        ops.append(("render", fr))
        if rng.random() < 0.7:
            ops.append(("releases", np.where(rng.random(V) < 0.5, s2.NO_RELEASE,
                                             rng.integers(0, 40000, V)).astype(np.uint32)))
        idx = rng.integers(0, V, max(1, V // 10)).astype(np.uint32)
        ds = np.zeros(idx.size, dtype=s2.VOICE_DESC)
        for j, i in enumerate(idx):
            ds[j] = _bank(8, int(kinds[i]), seed + j)[j % 8]
        ds["active"] = 1
        ops.append(("voices", idx, ds))
    ops.append(("render", 2048))
    return ops


def _apply(target, op, meters=None):
    if op[0] == "render":
        if isinstance(target, Twin):
            return target.render(op[1])
        return render_mixed(target, op[1], meters, canary=True)[0]
    if op[0] == "releases":
        target.set_releases(op[1])
    elif op[0] == "voices":
        target.set_voices(op[1], op[2])
    return None


@pytest.mark.parametrize("V", (33, 1000, 8192))
def test_pipelined_edits_match_default_mode_and_twin(V):
    voices, kinds = mixed_voices(V, seed=300 + V)
    ops = _edit_script(V, 300 + V, voices, kinds)
    runs = {}
    for n_sub in (1, 2, 4, 8):
        # entries past the voices must keep their values (off-by-one indices; padding never indexes a meter)
        guard = torch.full((V + 8,), -1.0, device="cuda", dtype=torch.float64)
        peak = torch.full((V + 8,), -1.0, device="cuda", dtype=torch.float32)
        guard[:V] = 0.0
        peak[:V] = 0.0
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
            bank.set_pipeline(n_sub)
            rows = [r for r in (_apply(bank, op, (guard.data_ptr(), peak.data_ptr())) for op in ops) if r is not None]
            bank.sync()
            runs[n_sub] = (rows, bank.get_state(), guard.clone(), peak.clone())
        assert torch.all(guard[V:] == -1.0) and torch.all(peak[V:] == -1.0), "meters written past the voices"
    for n_sub in (2, 4, 8):
        for a, b in zip(runs[1][0], runs[n_sub][0]):
            same(b, a, f"V={V} rows n_sub={n_sub}")
        for i in (1, 2, 3):
            same(runs[n_sub][i], runs[1][i], f"V={V} n_sub={n_sub} item {i}")
    twin = Twin(voices, kinds)
    try:
        rows = [r for r in (_apply(twin, op) for op in ops) if r is not None]
        for a, b in zip(rows, runs[1][0]):
            same(b, a, f"V={V} rows against the single-kind banks")
        same(runs[1][1], twin.get_state(), f"V={V} state against the single-kind banks")
        s, p = twin.meter_values()
        same(runs[1][2][:V], s, "sum_sq against the single-kind banks")
        same(runs[1][3][:V], p, "peak against the single-kind banks")
    finally:
        twin.close()


# ------------------------------------------------------------------------------ 5. per-voice edits

@pytest.mark.parametrize("V", (7, 333))
def test_edits_match_single_kind_banks(V):
    voices, kinds = mixed_voices(V, seed=400 + V)
    rng = np.random.default_rng(V)
    twin = Twin(voices, kinds)
    try:
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
            same(bank.filter_kinds, kinds, "filter_kinds")
            for step in range(4):
                fr = 1000 + 17 * step
                same(render_mixed(bank, fr)[0], twin.render(fr, metered=False), f"step {step}: rows")
                i = int(rng.integers(V))
                d = _bank(4, int(kinds[i]), 500 + step)[step:step + 1].copy()
                d["active"] = 1
                for t in (bank, twin):
                    t.set_voice(i, d)
                j = int(rng.integers(V))
                for t in (bank, twin):
                    t.release_voice(j)
                idx = rng.integers(0, V, 5).astype(np.uint32)
                ds = np.concatenate([_bank(4, int(kinds[x]), 600 + step)[:1] for x in idx])
                for t in (bank, twin):
                    t.set_voices(idx, ds)
                table = rng.integers(0, 30000, V).astype(np.uint32)
                for t in (bank, twin):
                    t.set_releases(table)
                if step == 2:
                    st = bank.get_state()
                    same(st, twin.get_state(), "state")
                    st["phase"] = rng.random(V).astype(np.float32)
                    for t in (bank, twin):
                        t.set_state(st)
            same(bank.get_state(), twin.get_state(), "final state")
    finally:
        twin.close()


def test_damping_is_validated_by_each_voice_kind():
    v = bankgen.make_bank(4, 64)
    kinds = np.array([s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP, s2.FILTER_FIRST_ORDER_LP, s2.FILTER_BIQUAD_BP], np.uint32)
    bad = v.copy()
    bad["damping"][1] = 0.0
    with pytest.raises(s2.S2Error):
        s2.VoiceBank.mixed(bad, kinds, SR)
    ok = v.copy()
    ok["damping"][[0, 2]] = 0.0
    with s2.VoiceBank.mixed(ok, kinds, SR) as bank:
        z = v[:1].copy()
        z["damping"] = 0.0
        bank.set_voice(0, z)                           # one-pole voice: accepted
        bank.set_voices(np.array([2], np.uint32), z)   # first-order voice: accepted
        for i in (1, 3):
            with pytest.raises(s2.S2Error):
                bank.set_voice(i, z)
            with pytest.raises(s2.S2Error):
                bank.set_voices(np.array([0, i], np.uint32), np.concatenate([z, z]))
        same(bank.filter_kinds, kinds, "filter_kinds")
    with s2.VoiceBank(v, SR, s2.FILTER_BIQUAD_HP) as single:
        same(single.filter_kinds, np.full(4, s2.FILTER_BIQUAD_HP, np.uint32), "single-kind filter_kinds")


# ------------------------------------------------------------------------------ 6. oracle

def test_small_mixed_bank_against_the_oracle():
    V = 96
    voices, kinds = mixed_voices(V, seed=7)
    frames = (1000, 2051)
    with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
        got = torch.cat([render_mixed(bank, fr)[0] for fr in frames], dim=1).cpu().numpy()
    for k in np.unique(kinds):
        m = kinds == k
        ref, _, _ = oracle_bank_render(voices[m], int(k), frames)
        assert_parity(ref, got[m], f"filter kind {k}")


# ------------------------------------------------------------------------------ 7. refusals, traces, launches

def test_time_split_is_refused_with_several_kinds():
    voices, kinds = mixed_voices(64, seed=8)
    with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
        with pytest.raises(s2.S2Error):
            bank.set_time_split(True)
    one = np.full(64, s2.FILTER_BIQUAD_LP, np.uint32)
    v = _bank(64, s2.FILTER_BIQUAD_LP, 8)
    with s2.VoiceBank.mixed(v, one, SR) as bank:
        bank.set_time_split(True)                      # one kind: the single-kind rule applies


@pytest.mark.parametrize("n_sub", (1, 4))
def test_trace_matches_single_kind_banks(n_sub):
    V = 333
    voices, kinds = mixed_voices(V, seed=9)
    twin = Twin(voices, kinds)
    try:
        with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
            bank.set_pipeline(n_sub)
            for fr in (1000, 2048):
                ph = torch.full((V, fr), float("nan"), device="cuda")
                bank.trace_phase(fr, ph, fr)
                same(ph, twin.trace(fr), f"trace of {fr} frames")
    finally:
        twin.close()


def test_validation_failures_create_nothing():
    v = bankgen.make_bank(40, 64)
    kinds = np.zeros(40, np.uint32)
    lib = s2.lib()
    h = C.c_void_p(1234)
    bad_kinds = kinds.copy()
    bad_kinds[39] = 6
    bad_voice = v.copy()
    bad_voice["pitch_hz"][5] = -1.0
    for vv, kk in ((v, bad_kinds), (v, None), (bad_voice, kinds)):
        rc = lib.s2_bank_create_mixed(0, SR, 40, _lib.ptr(vv), _lib.ptr(kk), None, C.byref(h))
        assert rc == _lib.S2_ERR_INVALID and not h.value
        h = C.c_void_p(1234)
    with pytest.raises(ValueError):
        s2.VoiceBank.mixed(v, kinds[:39], SR)


def _launches(fn, *args):
    n0 = s2.lib().s2_launch_count()
    fn(*args)
    return s2.lib().s2_launch_count() - n0


@pytest.mark.parametrize("V,n_sub", [(V, n) for V in (7, 32, 33, 2048, 65536) for n in (1, 2, 8)])
def test_launches_match_a_single_kind_bank(V, n_sub):
    """The launches of a single-kind bank of the same width and mode.  Exceptions: a multi-kind bank of up to 32
    voices adds its bus from the rows (one more launch when a bus is asked for), and in the pipelined mode a narrow
    bank's padding slots may fill more voice ranges (one launch each)."""
    T = 4096
    voices, kinds = mixed_voices(V, seed=10 + V)
    rows = torch.empty((V, T), device="cuda")
    bus = torch.empty(T, device="cuda")
    counts = []
    for make in (lambda: s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE), lambda: s2.VoiceBank.mixed(voices, kinds, SR)):
        with make() as bank:
            bank.set_pipeline(n_sub)
            counts.append([_launches(bank.render, T, r, T if r is not None else 0, b)
                           for r, b in ((rows, None), (None, bus), (rows, bus))])
            bank.sync()
    single, mixed = counts
    extra_ranges = 0
    if n_sub > 1:
        def ranges(S):
            groups = -(-S // 64)
            bounds = [min(groups * k // n_sub * 64, S) for k in range(n_sub + 1)]
            return sum(1 for k in range(n_sub) if bounds[k] < bounds[k + 1])
        extra_ranges = ranges(n_slots(kinds)) - ranges(V)
    extra_mix = 1 if V <= 32 and len(np.unique(kinds)) > 1 else 0
    assert mixed == [single[0] + extra_ranges, single[1] + extra_ranges + extra_mix,
                     single[2] + extra_ranges + extra_mix], (single, mixed)
    if V >= 2048:
        assert mixed == single


def test_mixed_sweep_bank_renders_finite():
    """bankgen's config-5 sweep over the six filter kinds: every kind present, every output finite."""
    voices, kinds = bankgen.make_mixed_sweep_bank(0, 96000, 0, 2048)
    assert set(np.unique(kinds)) == set(KINDS)
    sum_sq, peak = _meters(2048)
    with s2.VoiceBank.mixed(voices, kinds, SR) as bank:
        for _ in range(24):
            bank.render(4096, None, 0, None, sum_sq, peak)
        bank.sync()
    assert torch.all(torch.isfinite(sum_sq)) and torch.all(torch.isfinite(peak)) and torch.all(peak > 0)
