"""Note-ons in the streaming loop: K set_voice calls against one set_voices batch per step.

The shape of bench.py's e2e pass: 65,536 voices from bankgen (second-order low-pass), pipeline 4, 4,096-frame steps
from note-on; every step uploads the note-off table, then restarts K voices chosen from a seed, then renders into a
device ring with render_bus_host_async into two pinned buffers in flight (the host waits for and reads step i-1
after enqueueing step i).  Arm A applies the note-ons with K s2_bank_set_voice calls, arm B with one
s2_bank_set_voices.  Each (round, K) runs both arms on new banks, alternating, in one process; both must give the
same bus bytes at every step.  One JSON line per (arm, K):

    step_ms            median over steps and rounds of the time between consecutive step events (CUDA events)
    voice_samples_per_s  V * frames / the run's time (the larger of event time and wall clock), median over rounds
    note_on_host_us    median host time of the step's note-on call(s)

    python tools/bench_note_on.py [--steps 20] [--rounds 3] [--ks 0,66,655,6554]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import synth2_b200 as s2  # noqa: E402
from synth2_b200 import bankgen  # noqa: E402

SR = 48000
RENDER_FRAMES = 60 * SR


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = ""
    return name, out or "unknown"


def run(arm, K, args, voices, ring, stream):
    """One run from note-on; returns (step event times in ms, run time in s, note-on host times in s, buses)."""
    V, T = args.voices, args.block
    rng = np.random.default_rng(args.seed + K)
    rel_host = torch.from_numpy(voices["release_offset"].astype(np.uint32).view(np.int32)).pin_memory()
    bus_host = [torch.empty(T, dtype=torch.float32).pin_memory() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    buses, host_s = [], []
    fresh = voices.copy()
    fresh["active"] = 1
    fresh["frame_offset"] = 0
    with s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, stream=stream) as bank:
        bank.set_pipeline(args.pipeline)
        if K:
            # the same note-ons the bank already holds: a no-op that sizes the staging buffers before the timed steps
            idx = np.arange(K, dtype=np.uint32)
            if arm == "B":
                bank.set_voices(idx, voices[idx])
            else:
                for i in idx:
                    bank.set_voice(int(i), voices[i:i + 1])
        bank.sync()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev[0].record(stream)
        for i in range(args.steps):
            bank.set_releases(rel_host)
            if K:
                idx = rng.choice(V, K, replace=False).astype(np.uint32)
                descs = fresh[idx]
                h0 = time.perf_counter()
                if arm == "B":
                    bank.set_voices(idx, descs)
                else:
                    for j, v in enumerate(idx):
                        bank.set_voice(int(v), descs[j:j + 1])
                host_s.append(time.perf_counter() - h0)
            bank.render_bus_host_async(T, bus_host[i & 1], ring[i & 1], T)
            done[i & 1].record(stream)
            ev[i + 1].record(stream)
            if i > 0:
                done[(i - 1) & 1].synchronize()
                buses.append(bus_host[(i - 1) & 1].numpy().copy())
        done[(args.steps - 1) & 1].synchronize()
        buses.append(bus_host[(args.steps - 1) & 1].numpy().copy())
        bank.join(stream)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    return step_ms, max(ev[0].elapsed_time(ev[-1]) * 1e-3, wall), host_s, buses


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--voices", type=int, default=65536)
    ap.add_argument("--block", type=int, default=4096)
    ap.add_argument("--pipeline", type=int, default=4)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--ks", default="0,66,655,6554")
    ap.add_argument("--seed", type=int, default=1)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_note_on.py needs a CUDA device")
    ks = [int(k) for k in args.ks.split(",")]
    stream = torch.cuda.current_stream()
    voices = bankgen.make_bank(args.voices, RENDER_FRAMES, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    ring = [torch.empty((args.voices, args.block), device="cuda", dtype=torch.float32) for _ in range(2)]
    name, power = gpu_info()
    for arm in ("A", "B"):                                     # warm-up: modules, pinned buffers, allocator
        run(arm, ks[-1], argparse.Namespace(**{**vars(args), "steps": 3}), voices, ring, stream)
    res = {(arm, K): {"step_ms": [], "rate": [], "host": []} for K in ks for arm in ("A", "B")}
    for _ in range(args.rounds):
        for K in ks:
            first = None
            for arm in ("A", "B"):
                step_ms, secs, host_s, buses = run(arm, K, args, voices, ring, stream)
                r = res[(arm, K)]
                r["step_ms"] += step_ms
                r["rate"].append(args.voices * args.block * args.steps / secs)
                r["host"] += host_s
                if first is None:
                    first = buses
                else:
                    for i, (a, b) in enumerate(zip(first, buses)):
                        assert a.tobytes() == b.tobytes(), f"K={K}: arms differ at step {i}"
    for K in ks:
        for arm in ("A", "B"):
            r = res[(arm, K)]
            print(json.dumps({
                "arm": "set_voice x K" if arm == "A" else "set_voices", "K": K, "voices": args.voices,
                "block": args.block, "pipeline": args.pipeline, "steps": args.steps, "rounds": args.rounds,
                "step_ms": float(np.median(r["step_ms"])),
                "voice_samples_per_s": float(np.median(r["rate"])),
                "note_on_host_us": float(np.median(r["host"]) * 1e6) if r["host"] else 0.0,
                "gpu": name, "power_limit": power}), flush=True)


if __name__ == "__main__":
    main()
