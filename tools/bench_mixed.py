"""Mixed-filter banks (s2_bank_create_mixed) against one bank per filter kind, on one GPU.

Workload: config 5's share with the filter kind as a fourth axis (bankgen.make_mixed_sweep_bank(0, 10 s): 32,768
variants, each (cutoff, damping) cell of 32 detunes on one of the six kinds, ~5,461 voices per kind), the first 2 s in
4,096-frame blocks, every bank on one stream (no voice ranges), with rows (every variant's render kept on the device,
12.6 GB) and without (nothing stored).

  mixed        one bank of every kind: one launch per block
  mixed_pipe4  the same mixed bank in the pipelined mode with 4 voice ranges (s2_bank_set_pipeline)
  serial       six single-kind banks, one after another on one stream: six launches per block
  six_streams  the same six banks, each on its own stream; the host enqueues block by block
  kind_<k>     the single-kind bank of filter kind k alone (what each kind costs)

The rows of `mixed` are checked against those of the six banks, bit for bit.  Arms alternate inside each round and
every arm starts from the banks' initial state.  Prints one JSON document and writes it to --out.
`PYTHONPATH=. python tools/bench_mixed.py [--rounds 3] [--out profiles/mixed_b200.json]`
"""
import argparse
import json
import pathlib
import statistics
import subprocess

import numpy as np
import torch

import synth2_b200 as s2
from synth2_b200 import bankgen

SR = 48000
T = 4096


def gpu_info():
    q = "name,power.limit,clocks.max.sm"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    line = r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else ""
    return {"query": q, "nvidia_smi": line, "torch_name": torch.cuda.get_device_name()}


def summary(samples, voice_samples):
    med = statistics.median(samples)
    return {"seconds": samples, "median_s": med, "voice_samples_per_s": voice_samples / med}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=str(pathlib.Path(__file__).resolve().parent.parent / "profiles" / "mixed_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mixed.py needs a CUDA device")
    main_stream = torch.cuda.current_stream()
    V, total = bankgen.SWEEP_VARIANTS, 2 * SR
    voices, kinds = bankgen.make_mixed_sweep_bank(0, 10 * SR)
    # the six banks' voices in kind order: bank k's rows are a contiguous slice of the same [V, total] buffer
    order = np.argsort(kinds, kind="stable")
    groups = [(int(k), order[kinds[order] == k]) for k in range(bankgen.SWEEP_FILTER_KINDS)]
    streams = [torch.cuda.Stream() for _ in groups]
    mixed = s2.VoiceBank.mixed(voices, kinds, SR, stream=main_stream)
    mixed_pipe = s2.VoiceBank.mixed(voices, kinds, SR, stream=main_stream)
    mixed_pipe.set_pipeline(4)
    serial = [s2.VoiceBank(voices[m], SR, k, stream=main_stream) for k, m in groups]
    parallel = [s2.VoiceBank(voices[m], SR, k, stream=st) for (k, m), st in zip(groups, streams)]
    out = torch.empty((V, total), device="cuda", dtype=torch.float32)                   # 12.6 GB
    starts = np.cumsum([0] + [m.size for _, m in groups])
    states = {id(b): b.get_state() for b in [mixed, mixed_pipe, *serial, *parallel]}
    group_of = {id(b): i for banks in (serial, parallel) for i, b in enumerate(banks)}   # a kind bank's row slice

    def render_blocks(banks, rows):
        pos = 0
        while pos < total:
            fr = min(T, total - pos)
            for b in banks:
                if rows:
                    i = group_of.get(id(b))
                    r = out[:, pos:] if i is None else out[starts[i]:starts[i + 1], pos:]
                    b.render(fr, r, total)
                else:
                    b.render(fr)
            pos += fr

    def timed(banks, rows):
        for b in banks:
            b.set_state(states[id(b)])
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record(main_stream)
        for st in streams:
            st.wait_event(ev0)
        render_blocks(banks, rows)
        for b in banks:
            b.join(main_stream)
        for st in streams:
            main_stream.wait_stream(st)
        ev1.record(main_stream)
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) * 1e-3

    arms = {"mixed": [mixed], "mixed_pipe4": [mixed_pipe], "serial": serial, "six_streams": parallel}
    arms.update({f"kind_{k}": [b] for (k, _), b in zip(groups, serial)})
    for rows in (True, False):                       # warm-up of every shape the timed window uses
        for banks in arms.values():
            timed(banks, rows)
    timed([mixed], True)
    ref = out.clone()
    timed(serial, True)
    grouped = out[torch.from_numpy(np.argsort(order)).cuda()]      # six banks' rows back in voice order
    bits_equal = bool(torch.equal(ref.view(torch.int32), grouped.view(torch.int32)))
    del ref, grouped
    torch.cuda.empty_cache()

    res = {"gpu": gpu_info(), "rounds": args.rounds,
           "workload": "config 5 share with the filter kind as a fourth axis: 32,768 variants over six kinds "
                       f"({', '.join(str(m.size) for _, m in groups)} voices), first 2 s in 4,096-frame blocks, "
                       "one stream per bank, no voice ranges but in mixed_pipe4",
           "mixed_rows_equal_six_banks_rows": bits_equal}
    vs = V * total
    for rows in (True, False):
        samples = {name: [] for name in arms}
        for _ in range(args.rounds):
            for name, banks in arms.items():
                samples[name].append(timed(banks, rows))
        key = "rows" if rows else "no_rows"
        res[key] = {name: summary(s, vs) for name, s in samples.items()}
        med = {name: statistics.median(s) for name, s in samples.items()}
        res[key]["serial_over_mixed"] = med["serial"] / med["mixed"]
        res[key]["six_streams_over_mixed"] = med["six_streams"] / med["mixed"]
        res[key]["sum_of_kinds_over_serial"] = sum(med[f"kind_{k}"] for k, _ in groups) / med["serial"]
    for b in [mixed, mixed_pipe, *serial, *parallel]:
        b.close()
    text = json.dumps(res, indent=1)
    print(text)
    path = pathlib.Path(args.out)
    path.parent.mkdir(parents=True, exist_ok=True)
    path.write_text(text + "\n")


if __name__ == "__main__":
    main()
