"""Per-voice meters (s2_bank_render_metered) against rows kept on the device, on one GPU.

  config 5   one GPU's share of the sweep (bankgen.make_sweep_bank(0, 10 s), 32,768 variants, second-order low-pass,
             4 voice ranges), the first 2 s in 4,096-frame blocks as bench.py's extra_config5:
               rows     every variant's render kept on the device (12.6 GB), then the per-variant RMS in torch as
                        tools/measure_configs.py reads it (float64, 1,024 variants at a time); both timed
               meters   meters only: no per-voice stores
               both     rows and meters
             The RMS of `meters` is checked against that of `rows` (1e-6 relative) and its peaks against max |rows|
             (bit for bit).
  config 3   the bench bank (bankgen.make_bank(65,536), second-order low-pass, 4 voice ranges), 20 blocks of 4,096
             frames into a ring of two 1 GiB buffers: rows against rows + meters, the price of metering while the
             rows are written.

Arms alternate inside each round; every arm starts from the bank's initial state.  Prints one JSON document and
writes it to --out.  `PYTHONPATH=. python tools/bench_meters.py [--rounds 3] [--out profiles/meters_b200.json]`
"""
import argparse
import json
import pathlib
import statistics
import subprocess

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


def timed(stream, bank, body):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    body()
    bank.join(stream)
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) * 1e-3


def summary(samples, voice_samples):
    med = statistics.median(samples)
    return {"seconds": samples, "median_s": med, "voice_samples_per_s": voice_samples / med}


def config5(stream, rounds):
    V, total = bankgen.SWEEP_VARIANTS, 2 * SR
    voices = bankgen.make_sweep_bank(0, 10 * SR)
    bank = s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, stream=stream)
    bank.set_pipeline(4)
    out = torch.empty((V, total), device="cuda", dtype=torch.float32)                 # 12.6 GB
    sum_sq = torch.zeros(V, device="cuda", dtype=torch.float64)
    peak = torch.zeros(V, device="cuda", dtype=torch.float32)
    rms_rows = torch.empty(V, device="cuda", dtype=torch.float64)
    st = bank.get_state()
    for i in range(3):
        bank.render(T, out[:, i * T:], total, None, sum_sq, peak)
    bank.sync()

    def render(rows, meters):
        pos = 0
        while pos < total:
            fr = min(T, total - pos)
            bank.render(fr, out[:, pos:] if rows else None, total if rows else 0, None,
                        sum_sq if meters else None, peak if meters else None)
            pos += fr

    def rms_pass():
        for a in range(0, V, 1024):
            rms_rows[a:a + 1024] = out[a:a + 1024].double().pow(2).mean(dim=1).sqrt()

    arms = {"rows": [], "rows_render_only": [], "meters": [], "both": []}
    for _ in range(rounds):
        for arm in ("rows", "meters", "both"):
            bank.set_state(st)
            sum_sq.zero_()
            peak.zero_()
            if arm == "rows":
                t_render = timed(stream, bank, lambda: render(True, False))
                t_rms = timed(stream, bank, rms_pass)
                arms["rows"].append(t_render + t_rms)
                arms["rows_render_only"].append(t_render)
            else:
                arms[arm].append(timed(stream, bank, lambda: render(arm == "both", True)))
            if arm == "meters":
                meters_only = (sum_sq.clone(), peak.clone())
    # rms_rows is the last "rows" arm's RMS pass; `out` holds the rows of the last "both" arm (the same frames from the
    # same state: the same bits as the "rows" arm's)
    rms_meters = (meters_only[0] / total).sqrt()
    rel = float(((rms_meters - rms_rows).abs() / rms_rows.abs().clamp_min(1e-300)).max())
    same_bits = bool(torch.equal(meters_only[0].view(torch.int64), sum_sq.view(torch.int64))
                     and torch.equal(meters_only[1].view(torch.int32), peak.view(torch.int32)))
    peak = meters_only[1]
    peak_ok = True
    for a in range(0, V, 1024):
        want = (out[a:a + 1024].view(torch.int32) & 0x7fffffff).max(dim=1).values
        peak_ok &= bool(torch.equal(peak[a:a + 1024].view(torch.int32), want))
    bank.close()
    del out
    torch.cuda.empty_cache()
    vs = V * total
    return {"workload": "config 5 share: 32,768 sweep variants, biquad low-pass, 4 voice ranges, first 2 s in 4,096-frame "
                        "blocks",
            "rows_then_torch_rms": summary(arms["rows"], vs), "rows_render_only": summary(arms["rows_render_only"], vs),
            "meters_only": summary(arms["meters"], vs), "rows_and_meters": summary(arms["both"], vs),
            "rms_max_rel_diff_meters_vs_rows": rel, "peak_bits_equal_max_abs_rows": peak_ok,
            "meter_bits_meters_only_equal_rows_and_meters": same_bits,
            "rms_min": float(rms_rows.min()), "rms_max": float(rms_rows.max())}


def config3(stream, rounds):
    V, blocks = 65536, 20
    voices = bankgen.make_bank(V, 60 * SR, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    bank = s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, stream=stream)
    bank.set_pipeline(4)
    ring = [torch.empty((V, T), device="cuda", dtype=torch.float32) for _ in range(2)]   # 2 x 1 GiB
    sum_sq = torch.zeros(V, device="cuda", dtype=torch.float64)
    peak = torch.zeros(V, device="cuda", dtype=torch.float32)
    st = bank.get_state()
    for i in range(3):
        bank.render(T, ring[i & 1], T, None, sum_sq, peak)
    bank.sync()
    arms = {"rows": [], "rows_and_meters": []}
    for _ in range(rounds):
        for arm in arms:
            bank.set_state(st)
            m = arm == "rows_and_meters"
            arms[arm].append(timed(stream, bank, lambda: [bank.render(T, ring[i & 1], T, None, sum_sq if m else None,
                                                                      peak if m else None) for i in range(blocks)]))
    bank.close()
    vs = V * blocks * T
    r, m = statistics.median(arms["rows"]), statistics.median(arms["rows_and_meters"])
    return {"workload": "config 3 bench bank: 65,536 voices, biquad low-pass, 4 voice ranges, 20 blocks of 4,096 frames",
            "rows": summary(arms["rows"], vs), "rows_and_meters": summary(arms["rows_and_meters"], vs),
            "meters_cost": m / r - 1.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=str(pathlib.Path(__file__).resolve().parent.parent / "profiles" / "meters_b200.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_meters.py needs a CUDA device")
    stream = torch.cuda.current_stream()
    res = {"gpu": gpu_info(), "rounds": args.rounds, "config5": config5(stream, args.rounds),
           "config3": config3(stream, args.rounds)}
    text = json.dumps(res, indent=1)
    print(text)
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(text + "\n")


if __name__ == "__main__":
    main()
