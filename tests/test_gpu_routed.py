"""Routed voice banks (s2_bank_create_routed): every voice mixes into one of many mono buses, all summed by one render.

Bus g of a routed bank is specified as the d_bus_out of a mixed bank made from bus g's voices alone.  So, as in
test_gpu_mixed.py, a twin of standalone banks (one VoiceBank.mixed per non-empty bus) receives the same calls with voice
indices mapped into each bank, and every bus, row, meter and carried state must match it byte for byte (the sign of a
zero included).  The twins render in the default mode: a standalone bank's bus has the same bits in the default and
pipelined modes, so one twin checks the routed bank in every mode.
"""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import synth2_b200 as s2  # noqa: E402
from busref import U, closed_bus, closed_form, closed_rows, exact_bank, reference_order_bus  # noqa: E402
from synth2_b200 import _lib, bankgen  # noqa: E402

SR = 48000
KINDS = (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP, s2.FILTER_BIQUAD_HP, s2.FILTER_BIQUAD_BP,
         s2.FILTER_FIRST_ORDER_LP, s2.FILTER_FIRST_ORDER_HP)
FRAMES = (17, 64, 1000, 2051, 4096)


def _stride(fr):
    return (fr + 3) & ~3


def _meters(V):
    return (torch.zeros(V, device="cuda", dtype=torch.float64), torch.zeros(V, device="cuda", dtype=torch.float32))


def same(a, b, what):
    a = a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)
    b = b.cpu().numpy() if hasattr(b, "cpu") else np.asarray(b)
    assert a.shape == b.shape, what
    assert a.tobytes() == b.tobytes(), f"{what}: {np.sum(a.view(np.uint8) != b.view(np.uint8))} bytes differ"


def routing(sizes, seed):
    """bus_of_voice for buses of the given sizes, the voices of each bus scattered over the bank."""
    rng = np.random.default_rng(seed)
    return rng.permutation(np.repeat(np.arange(len(sizes)), sizes)).astype(np.uint32)


def routed_voices(sizes, n_kinds, seed, kind=None):
    """Voices for buses of `sizes`: drawn from test_gpu_edits's banks (all oscillator kinds, noise, cutoff followers,
    resting cutoffs, inactive voices), with random kinds out of the first n_kinds (or all `kind`)."""
    from test_gpu_mixed import mixed_voices
    V = int(sum(sizes))
    if kind is not None:
        from test_gpu_edits import _bank
        voices, kinds = _bank(V, kind, seed), np.full(V, kind, np.uint32)
    else:
        voices, kinds = mixed_voices(V, seed, n_kinds)
    return voices, kinds, routing(sizes, seed)


class Twin:
    """One standalone bank per non-empty bus of a routed bank, driven as one bank: voice i of the routed bank is voice
    local[i] of banks[buses[i]]."""

    def __init__(self, voices, kinds, buses, n_buses, time_split=False):
        self.V, self.n_buses = voices.shape[0], n_buses
        self.buses = buses
        self.members = {g: np.flatnonzero(buses == g) for g in range(n_buses) if np.any(buses == g)}
        self.local = np.zeros(self.V, dtype=np.int64)
        for m in self.members.values():
            self.local[m] = np.arange(m.size)
        self.banks = {g: s2.VoiceBank.mixed(voices[m], kinds[m], SR) for g, m in self.members.items()}
        self.meters = {g: _meters(m.size) for g, m in self.members.items()}
        self.index = {g: torch.from_numpy(m).cuda() for g, m in self.members.items()}
        if time_split:
            for b in self.banks.values():
                b.set_time_split(True)

    def close(self):
        for b in self.banks.values():
            b.close()

    def render(self, fr, rows=True, metered=True):
        """Rows [V, fr] (or None) and buses [n_buses, fr] of one render."""
        out_rows = torch.empty((self.V, fr), device="cuda") if rows else None
        buses = torch.zeros((self.n_buses, fr), device="cuda")
        for g, m in self.members.items():
            out = torch.full((m.size, _stride(fr)), float("nan"), device="cuda") if rows else None
            bus = torch.full((fr,), float("nan"), device="cuda")
            self.banks[g].render(fr, out, _stride(fr) if rows else 0, bus, *(self.meters[g] if metered else (None, None)))
            if rows:
                out_rows[self.index[g]] = out[:, :fr]
            buses[g] = bus
        torch.cuda.synchronize()
        return out_rows, buses

    def time_split_blocks(self):
        return [b.time_split_blocks for b in self.banks.values()]

    def set_voice(self, i, d):
        self.banks[int(self.buses[i])].set_voice(int(self.local[i]), d)

    def set_voices(self, idx, ds):
        for g in self.members:
            sel = self.buses[idx] == g
            if np.any(sel):
                self.banks[g].set_voices(self.local[idx[sel]], ds[sel])

    def release_voice(self, i):
        self.banks[int(self.buses[i])].release_voice(int(self.local[i]))

    def set_releases(self, table):
        for g, m in self.members.items():
            self.banks[g].set_releases(np.ascontiguousarray(table[m]))

    def get_state(self):
        st = np.zeros(self.V, dtype=s2.VOICE_STATE)
        for g, m in self.members.items():
            st[m] = self.banks[g].get_state()
        return st

    def meter_values(self):
        s, p = np.zeros(self.V), np.zeros(self.V, dtype=np.float32)
        for g, m in self.members.items():
            s[m] = self.meters[g][0].cpu().numpy()
            p[m] = self.meters[g][1].cpu().numpy()
        return s, p


def render_routed(bank, fr, rows=True, meters=None):
    """Rows [V, fr] (or None) and buses [n_buses, fr] of one s2_bank_render_buses call.  The row buffer has one more
    row past the last voice, which must keep its value (a padding slot writes no row)."""
    V = bank.n_voices
    out = None
    if rows:
        out = torch.full((V + 1, _stride(fr)), float("nan"), device="cuda")
        out[V] = 7.0
    buses = torch.full((bank.n_buses, _stride(fr)), float("nan"), device="cuda")
    bank.render(fr, out, _stride(fr) if rows else 0, None, *(meters if meters is not None else (None, None)),
                buses=buses)
    bank.sync()
    if rows:
        assert torch.all(out[V] == 7.0), "a padding slot wrote past the caller's rows"
        out = out[:V, :fr]
    return out, buses[:, :fr]


def _desc(kind, seed, j):
    from test_gpu_edits import _bank
    d = _bank(8, int(kind), seed)[j % 8:j % 8 + 1].copy()
    d["active"] = 1
    return d


def _edit(rng, step, bank, twin, kinds, staged):
    """One round of edits, the same on the routed bank and the twin.  staged: only the note-off table (the next
    render is pipelined and applies it)."""
    V = bank.n_voices
    table = np.where(rng.random(V) < 0.5, s2.NO_RELEASE, rng.integers(0, 40000, V)).astype(np.uint32)
    if not staged:
        i = int(rng.integers(V))
        d = _desc(kinds[i], 700 + step, step)
        j = int(rng.integers(V))
        for t in (bank, twin):
            t.set_voice(i, d)
            t.release_voice(j)
    idx = rng.integers(0, V, max(1, V // 10)).astype(np.uint32)
    ds = np.concatenate([_desc(kinds[x], 800 + step, n) for n, x in enumerate(idx)])
    for t in (bank, twin):
        t.set_releases(table)
        t.set_voices(idx, ds)


# ------------------------------------------------------------------------------ 1. against standalone banks

CASES = {
    # bus widths 1 to 1,000 in one bank, one kind and six (multi-kind buses of up to 32 voices among them)
    "widths-one-kind": dict(sizes=[1, 7, 32, 33, 333, 1000], kind=s2.FILTER_BIQUAD_LP),
    "widths-six-kinds": dict(sizes=[1, 7, 32, 33, 333, 1000], n_kinds=6),
    # a bus of 16,384 voices (512 warps and more: the four-frames-per-lane reduction) next to narrow buses
    "wide-one-kind": dict(sizes=[16384, 7, 40], kind=s2.FILTER_ONE_POLE),
    "wide-six-kinds": dict(sizes=[5, 16384, 30, 100], n_kinds=6),
    # empty buses are +0.0
    "empty-buses": dict(sizes=[0, 5, 0, 40, 0], n_kinds=3),
    # 1,000 buses over 65,536 voices, and three empty ones
    "thousand-buses": dict(sizes=[65] * 464 + [66] * 536 + [0] * 3, n_kinds=6),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_buses_rows_meters_state_match_standalone_banks(case):
    c = CASES[case]
    voices, kinds, buses = routed_voices(c["sizes"], c.get("n_kinds", 1), seed=len(case), kind=c.get("kind"))
    n_buses = len(c["sizes"])
    V = voices.shape[0]
    rng = np.random.default_rng(len(case))
    big = V > 20000
    # (frames, voice ranges, rows, meters): every mode, with and without rows and meters
    plan = [(17, 1, True, True), (64, 2, False, True), (1000, 4, True, False), (2051, 8, False, False),
            (4096, 1, True, True), (4096, 4, False, True), (2051, 1, False, True), (1000, 2, True, True)]
    if big:
        plan = [(1000, 1, True, True), (4096, 4, False, True), (2051, 8, True, False), (4096, 1, False, False)]
    twin = Twin(voices, kinds, buses, n_buses)
    meters = _meters(V)
    try:
        with s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR) as bank:
            assert bank.n_buses == n_buses
            same(bank.bus_of_voice, buses, "bus_of_voice")
            same(bank.filter_kinds, kinds, "filter_kinds")
            for step, (fr, n_sub, rows, metered) in enumerate(plan):
                bank.set_pipeline(n_sub)
                if step and not big:
                    _edit(rng, step, bank, twin, kinds, staged=n_sub > 1)
                got_rows, got = render_routed(bank, fr, rows, meters if metered else None)
                want_rows, want = twin.render(fr, rows, metered)
                same(got, want, f"{case} step {step}: buses of {fr} frames, n_sub={n_sub} rows={rows}")
                if rows:
                    same(got_rows, want_rows, f"{case} step {step}: rows")
            same(bank.get_state(), twin.get_state(), f"{case}: state")
            s, p = twin.meter_values()
            same(meters[0], s, f"{case}: sum_sq")
            same(meters[1], p, f"{case}: peak")
            for g, size in enumerate(c["sizes"]):
                if size == 0:
                    assert torch.all(got[g].view(torch.int32) == 0), f"empty bus {g} is not +0.0"
    finally:
        twin.close()


@pytest.mark.gpu
def test_one_bus_is_a_mixed_bank():
    """n_buses = 1: the bank s2_bank_create_mixed makes, bus for bus (its d_bus_out) and row for row."""
    voices, kinds, _ = routed_voices([333], 6, seed=5)
    buses = np.zeros(333, np.uint32)
    with s2.VoiceBank.routed(voices, kinds, buses, 1, SR) as routed, s2.VoiceBank.mixed(voices, kinds, SR) as mixed:
        assert routed.n_buses == 1
        for n_sub in (1, 4):
            routed.set_pipeline(n_sub)
            mixed.set_pipeline(n_sub)
            for fr in FRAMES:
                rows, bus = render_routed(routed, fr)
                out = torch.full((333, _stride(fr)), float("nan"), device="cuda")
                b = torch.full((fr,), float("nan"), device="cuda")
                mixed.render(fr, out, _stride(fr), b)
                mixed.sync()
                same(bus[0], b, f"bus of {fr} frames, n_sub={n_sub}")
                same(rows, out[:, :fr], "rows")


# ------------------------------------------------------------------------------ 2. time-split mode

@pytest.mark.gpu
@pytest.mark.parametrize("fk", (s2.FILTER_ONE_POLE, s2.FILTER_BIQUAD_LP))
def test_time_split_buses_match_standalone_banks(fk):
    """Single-kind routed banks of up to 16,384 voices take time-split blocks; where the routed bank and every twin
    admitted the same block (admission is per bank), the buses match bit for bit.  Rows and state always do."""
    sizes = [1, 7, 32, 33, 500, 0]
    voices, kinds, buses = routed_voices(sizes, 1, seed=20 + fk, kind=fk)
    voices["mod_env_to_osc_freq"] = 0.0
    twin = Twin(voices, kinds, buses, len(sizes), time_split=True)
    compared = 0
    try:
        with s2.VoiceBank.routed(voices, kinds, buses, len(sizes), SR) as bank:
            bank.set_time_split(True)
            for fr in (4096, 1024, 2048, 1000, 4096, 8192):
                b0, t0 = bank.time_split_blocks, twin.time_split_blocks()
                got_rows, got = render_routed(bank, fr)
                want_rows, want = twin.render(fr, metered=False)
                same(got_rows, want_rows, f"rows of {fr} frames")
                ts = bank.time_split_blocks - b0
                if all(t1 - t == ts for t, t1 in zip(t0, twin.time_split_blocks())):
                    same(got, want, f"buses of {fr} frames (time-split: {ts})")
                    compared += ts
            same(bank.get_state(), twin.get_state(), "state")
    finally:
        twin.close()
    assert compared >= 2, "too few time-split blocks were compared"


# ------------------------------------------------------------------------------ 3. exact banks

@pytest.mark.gpu
@pytest.mark.parametrize("V", (40, 1000, 65536))
def test_exact_buses_equal_the_closed_form(V):
    """Exact banks (busref.exact_bank): every bus is the exact sum of its voices, whatever its width, in the default
    and pipelined modes; buses of up to 32 voices are the reference-order sum of their rows."""
    rng = np.random.default_rng(V)
    n_buses = max(2, V // 50)
    sizes = rng.multinomial(V - n_buses, np.ones(n_buses) / n_buses) + 1
    sizes[0], sizes[-1] = 3, 0
    sizes[1] += V - int(sizes.sum())
    buses = routing(sizes, V)
    voices = exact_bank(V, seed=V)
    kinds = np.zeros(V, np.uint32)
    n0 = voices["frame_offset"].astype(np.int64)
    fr = 4096
    with s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR) as bank:
        for n_sub in (1, 4, 1):
            bank.set_pipeline(n_sub)
            rows, got = render_routed(bank, fr, rows=V <= 1000)
            val, stop = closed_form(voices, n0, fr)
            got = got.cpu().numpy()
            for g in range(n_buses):
                m = buses == g
                same(got[g], closed_bus(val[m], stop[m], fr), f"V={V} n_sub={n_sub} bus {g} of {m.sum()} voices")
                if rows is not None and m.sum() <= 32:
                    same(got[g], reference_order_bus(closed_rows(val[m], stop[m], fr)), f"bus {g}: voice order")
            n0 = np.asarray(n0 + np.where(voices["active"] != 0, fr, 0))


# ------------------------------------------------------------------------------ 4. the whole-bank bus

def _bank_warps(kinds, buses, n_buses):
    """Warps of a routed bank: each bus laid out as a mixed bank of its voices (kind groups padded to whole warps but
    the last), each bus but the last non-empty one padded to whole warps."""
    slots = []
    for g in range(n_buses):
        k = kinds[buses == g]
        sizes = [int(np.sum(k == x)) for x in KINDS if np.any(k == x)]
        if sizes:
            slots.append(sum(-(-n // 32) * 32 for n in sizes[:-1]) + sizes[-1])
    return -(-(sum(-(-n // 32) * 32 for n in slots[:-1]) + slots[-1]) // 32)


@pytest.mark.gpu
@pytest.mark.parametrize("sizes", ([3, 4], [10, 22], [100, 200, 33], [1000, 7, 3000, 89]))
def test_whole_bank_bus(sizes):
    """s2_bank_render's d_bus_out on a routed bank: the voice-order sum up to 32 voices; above that within
    gamma_d * sum|rows| (d: 32 in a warp, at most, then the reduction over the bank's warps), the same in every mode."""
    voices, kinds, buses = routed_voices(sizes, 6, seed=sum(sizes))
    V, n_buses = voices.shape[0], len(sizes)
    R = _bank_warps(kinds, buses, n_buses)
    seen = {}
    for n_sub in (1, 2, 4, 8):
        with s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR) as bank:
            bank.set_pipeline(n_sub)
            for fr in (1000, 2051, 4096):
                out = torch.full((V, _stride(fr)), float("nan"), device="cuda")
                bus = torch.full((fr,), float("nan"), device="cuda")
                bank.render(fr, out, _stride(fr), bus)
                bank.sync()
                rows = out[:, :fr].double()
                if V <= 32:
                    same(bus, reference_order_bus(out[:, :fr].cpu().numpy()), f"V={V} bus of {fr} frames")
                else:
                    wide = R >= 512 and fr % 128 == 0
                    d = 32 + (-(-R // 64) + 11 if wide else -(-R // 32) + 9)
                    gamma = d * U / (1 - d * U)
                    err = (bus.double() - rows.sum(0)).abs()
                    assert torch.all(err <= gamma * rows.abs().sum(0)), f"V={V} {fr} frames: bus outside its bound"
                seen.setdefault(fr, []).append(bus.cpu().numpy())
    for fr, bs in seen.items():
        for b in bs[1:]:
            same(b, bs[0], f"bus of {fr} frames across modes")


# ------------------------------------------------------------------------------ 5. oracle

@pytest.mark.gpu
def test_sixteen_parts_against_the_oracle():
    """16 parts of 8 voices, each part its own patch and filter: each bus is the reference-order sum of the oracle's
    rows of its part, within the parity bar."""
    from test_gpu_edits import _bank
    from test_gpu_parity import assert_parity, oracle_bank_render
    parts = [_bank(8, KINDS[p % 6], 40 + p) for p in range(16)]
    voices = np.concatenate(parts)
    kinds = np.repeat([KINDS[p % 6] for p in range(16)], 8).astype(np.uint32)
    buses = routing([8] * 16, 3)
    order = np.argsort(buses, kind="stable")         # part p's voices, in voice order, are voices[buses == p]
    voices[order] = voices.copy()
    kinds[order] = kinds.copy()
    frames = (1000, 2051)
    with s2.VoiceBank.routed(voices, kinds, buses, 16, SR) as bank:
        got = torch.cat([render_routed(bank, fr, rows=False)[1] for fr in frames], dim=1).cpu().numpy()
    for p in range(16):
        m = buses == p
        ref, _, _ = oracle_bank_render(voices[m], int(kinds[m][0]), frames)
        assert_parity(reference_order_bus(ref), got[p], f"part {p}")


# ------------------------------------------------------------------------------ 6. launches, multi-GPU, arguments

def _launches(fn, *args, **kw):
    n0 = s2.lib().s2_launch_count()
    fn(*args, **kw)
    return s2.lib().s2_launch_count() - n0


@pytest.mark.gpu
@pytest.mark.parametrize("n_sub", (1, 4))
def test_reduction_launches_do_not_grow_with_the_buses(n_sub):
    """A bus of 16,384 voices (the four-frames-per-lane form) and n_buses - 1 buses of 8 voices of several kinds (the
    rows form) or of one (a copy): at most one launch per form, however many buses."""
    T = 4096
    counts = {}
    for n_buses in (4, 16, 256, 1000):
        sizes = [16384] + [8] * (n_buses - 1)
        voices, kinds, buses = routed_voices(sizes, 6, seed=n_buses)
        bs = torch.empty((n_buses, T), device="cuda")
        with s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR) as bank:
            bank.set_pipeline(n_sub)
            counts[n_buses] = (_launches(bank.render, T, None, 0, None, buses=bs),
                               _launches(bank.render, T, None, 0, None))
            bank.sync()
    renders = {n: c[1] for n, c in counts.items()}
    extra = {n: c[0] - c[1] for n, c in counts.items()}
    assert all(1 <= e <= 3 for e in extra.values()), counts
    assert max(renders.values()) <= n_sub, counts


@pytest.mark.gpu
def test_reduce_bus_of_contiguous_buses_single_rank():
    """With bus_stride == frames the buses are one [n_buses][frames] array: one s2_bank_reduce_bus of frames * n_buses
    reduces them all (the identity on one rank, through real NCCL)."""
    from synth2_b200.shard import MasterBus
    T, n_buses = 4096, 12
    voices, kinds, buses = routed_voices([8] * n_buses, 6, seed=12)
    with s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR) as bank:
        bank.set_pipeline(2)
        bs = torch.zeros((n_buses, T), device="cuda")
        master = torch.full((n_buses, T), float("nan"), device="cuda")
        bank.render(T, None, 0, None, buses=bs)
        try:
            comm = MasterBus(0, 1, 0)
        except s2.S2Error as e:
            pytest.skip(f"NCCL not available: {e}")
        with comm:
            comm.reduce(bank, bs.view(-1), master.view(-1), root=0, stream=torch.cuda.current_stream())
            torch.cuda.synchronize()
        assert torch.equal(bs, master)
        assert float(bs.abs().max()) > 0.0


@pytest.mark.gpu
def test_render_buses_argument_checks():
    voices, kinds, buses = routed_voices([5, 40], 2, seed=1)
    lib = s2.lib()
    with s2.VoiceBank.routed(voices, kinds, buses, 2, SR) as bank:
        bs = torch.zeros((2, 256), device="cuda")
        sq, pk = _meters(45)
        h, p = bank._h, bs.data_ptr()
        cases = [(None, 64, p, 256, None, None), (h, 64, None, 256, None, None), (h, 64, p + 4, 256, None, None),
                 (h, 64, p, 130, None, None), (h, 256, p, 252, None, None), (h, 64, p, 256, sq.data_ptr(), None),
                 (h, 64, p, 256, None, pk.data_ptr())]
        for bh, fr, d, stride, s, pe in cases:
            rc = lib.s2_bank_render_buses(bh, fr, None, 0, _lib.ptr(d), stride, _lib.ptr(s), _lib.ptr(pe))
            assert rc == _lib.S2_ERR_INVALID, (fr, d, stride, s, pe)
        lib.s2_bank_sync(h)
        assert torch.all(bs == 0.0), "a refused call wrote"
        with pytest.raises(ValueError):
            bank.render(64, None, 0, None, buses=torch.zeros((3, 64), device="cuda"))
        with pytest.raises(ValueError):
            bank.render(64, None, 0, torch.zeros(64, device="cuda"), buses=bs)


def test_routed_argument_validation_happens_before_the_device():
    """Creation refuses bad routing before it touches a device, and s2_bank_render_buses checks its arguments before
    it reads the bank, so neither needs a GPU."""
    lib = s2.lib()
    v = bankgen.make_bank(4, 64)
    kinds = np.zeros(4, np.uint32)
    buses = np.array([0, 1, 2, 1], np.uint32)
    h = C.c_void_p(1234)
    for b, n in ((None, 3), (buses, 2), (buses, 0), (buses, _lib.MAX_BUSES + 1)):
        rc = lib.s2_bank_create_routed(0, SR, 4, _lib.ptr(v), _lib.ptr(kinds), _lib.ptr(b), n, None, C.byref(h))
        assert rc == _lib.S2_ERR_INVALID and not h.value, (b, n)
        h = C.c_void_p(1234)
    assert lib.s2_bank_buses(None, None, None) == _lib.S2_ERR_INVALID
    placeholder = np.zeros(64, np.uint8)            # never read: every check below fails first
    d = placeholder.ctypes.data
    al = (d + 15) & ~15
    for bank, buf, stride, fr, sq, pk in ((None, al, 64, 64, None, None), (d, None, 64, 64, None, None),
                                          (d, al + 4, 64, 64, None, None), (d, al, 66, 64, None, None),
                                          (d, al, 60, 64, None, None), (d, al, 64, 64, al, None),
                                          (d, al, 64, 64, None, al)):
        rc = lib.s2_bank_render_buses(_lib.ptr(bank), fr, None, 0, _lib.ptr(buf), stride, _lib.ptr(sq), _lib.ptr(pk))
        assert rc == _lib.S2_ERR_INVALID, (bank, buf, stride, fr, sq, pk)
