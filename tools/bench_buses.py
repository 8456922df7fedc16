"""Routed banks (s2_bank_create_routed, s2_bank_render_buses) against what a host can do without them, on one GPU.

Workloads:
  bench_<B>   the bench bank (bankgen.make_bank, 65,536 biquad low-pass voices) with voice i on bus i % B, B = 16 and
              256; the first 2 s in 4,096-frame blocks, pipelined with 4 voice ranges (the per-bus banks: each on its
              own stream, in the default mode)
  parts_16x8  a multitimbral host: 16 parts of 8 voices, part p on bus p with filter kind p % 6 (test_gpu_edits's
              voice mix), the first 2 s in 4,096-frame blocks, default mode

Arms (every arm starts from the banks' initial state; arms alternate inside each round; medians are reported):
  routed          one routed bank, s2_bank_render_buses: every bus, no rows
  mono            the same routed bank through s2_bank_render with d_bus_out: one bus, the floor of the reduction
  plain           (bench_*) a bank made by s2_bank_create from the same voices, s2_bank_render with d_bus_out: what
                  the per-warp kernel (render_kernel_mixed) costs a single-kind routed bank against render_kernel
  rows_index_add  a bank made by s2_bank_create (bench_*) or s2_bank_create_mixed (parts) writing every row, then torch
                  index_add_ of the rows into the buses: what a host does without routing.  This bank renders on the
                  caller's stream (no voice ranges): a pipelined bank's ranges do not wait for the caller's reads of the
                  row buffer, so the next block would overwrite rows the index_add has not read yet
  banks_streams   one bank per bus, each on its own stream, each writing its d_bus_out

The buses of `routed` are checked against those of `banks_streams`, bit for bit, over the whole window.
Prints one JSON document and writes it to --out.  `PYTHONPATH=. python tools/bench_buses.py [--rounds 3]`
"""
import argparse
import json
import pathlib
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import synth2_b200 as s2  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402

SR = 48000
T = 4096
TOTAL = 2 * SR


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"query": q, "nvidia_smi": line, "torch_name": torch.cuda.get_device_name()}


def slots_of(kinds, buses, n_buses):
    """Slots of a routed bank (s2_bank_create_routed's layout): each bus as a mixed bank of its voices, each bus but
    the last non-empty one padded to whole warps."""
    per_bus = []
    for g in range(n_buses):
        k = kinds[buses == g]
        sizes = [int(np.sum(k == x)) for x in range(6) if np.any(k == x)]
        if sizes:
            per_bus.append(sum(-(-n // 32) * 32 for n in sizes[:-1]) + sizes[-1])
    return sum(-(-n // 32) * 32 for n in per_bus[:-1]) + per_bus[-1]


def workload(name, voices, kinds, buses, n_buses, n_sub, single_kind, rounds):
    main = torch.cuda.current_stream()
    V = voices.shape[0]
    members = [np.flatnonzero(buses == g) for g in range(n_buses)]
    streams = [torch.cuda.Stream() for _ in members]
    routed = s2.VoiceBank.routed(voices, kinds, buses, n_buses, SR, stream=main)
    routed.set_pipeline(n_sub)
    if single_kind:
        plain = s2.VoiceBank(voices, SR, int(kinds[0]), stream=main)
    else:
        plain = s2.VoiceBank.mixed(voices, kinds, SR, stream=main)
    plain.set_pipeline(n_sub)
    rows_bank = (s2.VoiceBank(voices, SR, int(kinds[0]), stream=main) if single_kind
                 else s2.VoiceBank.mixed(voices, kinds, SR, stream=main))
    per_bus = [s2.VoiceBank.mixed(voices[m], kinds[m], SR, stream=st) for m, st in zip(members, streams)]
    bus_index = torch.from_numpy(buses.astype(np.int64)).cuda()
    buses_out = torch.zeros((n_buses, TOTAL), device="cuda")
    mono_out = torch.zeros(TOTAL, device="cuda")
    rows = torch.empty((V, T), device="cuda")
    states = {id(b): b.get_state() for b in [routed, plain, rows_bank, *per_bus]}

    def run(arm):
        pos = 0
        while pos < TOTAL:
            fr = min(T, TOTAL - pos)
            if arm == "routed":
                routed.render(fr, None, 0, None, buses=buses_out[:, pos:], bus_stride=TOTAL)
            elif arm == "mono":
                routed.render(fr, None, 0, mono_out[pos:])
            elif arm == "plain":
                plain.render(fr, None, 0, mono_out[pos:])
            elif arm == "rows_index_add":
                rows_bank.render(fr, rows, T)
                blk = buses_out[:, pos:pos + fr]
                blk.zero_()
                blk.index_add_(0, bus_index, rows[:, :fr])
            else:
                for g, b in enumerate(per_bus):
                    b.render(fr, None, 0, buses_out[g, pos:])
            pos += fr

    def timed(arm):
        banks = {"routed": [routed], "mono": [routed], "plain": [plain], "rows_index_add": [rows_bank]}.get(arm, per_bus)
        for b in banks:
            b.set_state(states[id(b)])
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(main)
        for st in streams:
            st.wait_event(ev0)
        run(arm)
        for b in banks:
            b.join(main)
        for st in streams:
            main.wait_stream(st)
        ev1.record(main)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) * 1e-3

    arms = ["routed", "mono", "plain", "rows_index_add", "banks_streams"]
    for arm in arms:                                     # warm-up of every shape the timed window uses
        timed(arm)
    timed("routed")
    ref = buses_out.clone()
    timed("banks_streams")
    bits_equal = bool(torch.equal(ref.view(torch.int32), buses_out.view(torch.int32)))
    timed("rows_index_add")
    err = float((buses_out.double() - ref.double()).abs().max())
    del ref
    samples = {arm: [] for arm in arms}
    for _ in range(rounds):
        for arm in arms:
            samples[arm].append(timed(arm))
    med = {arm: statistics.median(s) for arm, s in samples.items()}
    n_slots = slots_of(kinds, buses, n_buses)
    res = {"voices": V, "buses": n_buses, "voice_ranges": n_sub, "slots": n_slots, "padding_slots": n_slots - V,
           "routed_buses_equal_banks_streams": bits_equal, "rows_index_add_max_abs_diff_from_routed": err,
           "arms": {arm: {"seconds": s, "median_s": med[arm]} for arm, s in samples.items()},
           "routed_minus_mono_ms": (med["routed"] - med["mono"]) * 1e3,
           "mono_over_plain": med["mono"] / med["plain"],
           "rows_index_add_over_routed": med["rows_index_add"] / med["routed"],
           "banks_streams_over_routed": med["banks_streams"] / med["routed"]}
    for b in [routed, plain, rows_bank, *per_bus]:
        b.close()
    print(name, json.dumps({k: v for k, v in res.items() if k != "arms"}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "buses_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_buses.py needs a CUDA device")
    res = {"gpu": gpu_info(), "rounds": args.rounds, "block_frames": T, "window_frames": TOTAL}
    V = 65536
    voices = bankgen.make_bank(V, 60 * SR, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    kinds = np.full(V, s2.FILTER_BIQUAD_LP, np.uint32)
    for B in (16, 256):
        buses = (np.arange(V) % B).astype(np.uint32)
        res[f"bench_{B}"] = workload(f"bench_{B}", voices, kinds, buses, B, 4, True, args.rounds)
    from test_gpu_edits import _bank
    parts = [_bank(8, p % 6, 40 + p) for p in range(16)]
    pv = np.concatenate(parts)
    pv["frame_offset"] = 0
    pk = np.repeat(np.arange(16) % 6, 8).astype(np.uint32)
    pb = np.repeat(np.arange(16), 8).astype(np.uint32)
    res["parts_16x8"] = workload("parts_16x8", pv, pk, pb, 16, 1, False, args.rounds)
    text = json.dumps(res, indent=1)
    print(text)
    path = pathlib.Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(text + "\n")


if __name__ == "__main__":
    main()
