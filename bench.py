#!/usr/bin/env python3
"""bench.py — voice-samples/sec of the render hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE config 3, per GPU): 65,536 voices, oscillator + resonant biquad (2nd-order
low-pass) + ADSR, 48 kHz, 60 s = 2,880,000 frames per voice, streamed as 4,096-frame blocks through
a ring of two 1 GiB voice-major output buffers with the DSP state carried on the device.
One "step" = one block of every voice, FROM NOTE-ON: --steps K renders the first K * 4,096 frames of the
60 s render (the default 704 steps are the whole render; the last step is the 512-frame remainder).  The first
200 ms after note-on (2.3 steps) hold the mod-envelope sweep of the cutoff, the next ~1 s the attack / decay
ramps; `step_ms` in the result shows them.  N GPUs = N x 65,536 voices, each rank owning a contiguous voice
range ("weak").

  value      device-resident throughput: inputs (voice table, state) already in HBM, CUDA events
             around the K steps on the launching stream, max over ranks.
  step_ms    per-step completion intervals (CUDA events after every step, rank 0).
  parity     after the timed region: the CPU oracle renders a sample of the timed voices over the same frames;
             final oscillator phase bit-for-bit, max |err| and SNR of the last block.
  e2e        the same render driven through the host-buffer C-ABI calls a streaming caller uses:
             every step uploads the note-off table (pinned host -> device), renders the block
             (per-voice output stays in the device ring) with the mono mix, and copies the mix
             (the `Synth::sample` result) back to pinned host memory.
  extra      the other BASELINE configs on the same GPU(s): config 2 (1,024 voices, time-split), config 5
             (32,768 patch variants) at N = 1; config 4 (262,144 voices over N GPUs, master bus, one NCCL
             reduce) at N > 1.
  roofline   HBM: 4 algorithmic bytes per voice-sample (one f32 store, touched once; SURVEY 8d)
  cpu_baseline / --impl reference
             the CPU port of the reference path (oracle/, "port": the Rust reference cannot be
             built here) on all host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import pathlib
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

SR = 48000
VOICES_PER_GPU = 65536
BLOCK = 4096
RENDER_FRAMES = 60 * SR          # 2,880,000
DEFAULT_STEPS = (RENDER_FRAMES + BLOCK - 1) // BLOCK   # 704
FILTER_BIQUAD = 1
BYTES_PER_VOICE_SAMPLE = 4


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=DEFAULT_STEPS)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--voices", type=int, default=VOICES_PER_GPU, help="voices per GPU")
    ap.add_argument("--block", type=int, default=BLOCK)
    ap.add_argument("--master-bus", action="store_true",
                    help="N>1: also mix every rank's voices and NCCL-reduce the whole-render bus to rank 0 "
                         "(BASELINE config 4), inside the timed region")
    ap.add_argument("--pipeline", type=int, default=4,
                    help="render each GPU's bank as this many voice ranges on internal streams (1 = single stream)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config 2 / 4 / 5 measurements")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=30.0, help="target CPU time of the baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (float32, a fixed "
                         "sample of voices, at most 64 MiB in all) so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def step_frames(steps, block):
    """Frames of each step: 4,096 each; the default 704 steps end exactly at 60 s."""
    if block == BLOCK and steps == DEFAULT_STEPS:
        return [BLOCK] * (steps - 1) + [RENDER_FRAMES - BLOCK * (steps - 1)]
    return [block] * steps


# ------------------------------------------------------------------------------------------
# clocks

class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nv = None

    def _run(self):
        nv = self._nv
        names = {
            "nvmlClocksEventReasonHwSlowdown": "hw_slowdown",
            "nvmlClocksThrottleReasonHwSlowdown": "hw_slowdown",
            "nvmlClocksThrottleReasonHwThermalSlowdown": "hw_thermal_slowdown",
            "nvmlClocksThrottleReasonSwThermalSlowdown": "sw_thermal_slowdown",
            "nvmlClocksThrottleReasonSwPowerCap": "sw_power_cap",
            "nvmlClocksThrottleReasonHwPowerBrakeSlowdown": "hw_power_brake",
        }
        masks = {getattr(nv, k): v for k, v in names.items() if hasattr(nv, k)}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
                for m, name in masks.items():
                    if r & m:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.001)

    def __enter__(self):                      # re-enterable: the device-resident and the e2e timed regions both sample
        self._stop.clear()
        if self._nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------
# CPU arm: the port of the reference path (oracle/) on the host cores

_ORACLE_FLAGS = None


def cpu_oracle():
    """The C port of the reference path, built for this host (oracle/Makefile `native`)."""
    global _ORACLE_FLAGS
    sys.path.insert(0, str(ROOT / "tests"))
    import oracle
    if _ORACLE_FLAGS is None:
        _ORACLE_FLAGS = oracle.use_native_build()
    return oracle


def cpu_port_throughput(voices_desc, n_threads, frames, repeats=1):
    oracle = cpu_oracle()
    best = None
    for _ in range(repeats):
        st = oracle.bank_init_states(voices_desc)
        t0 = time.perf_counter()
        # per-thread scratch rows instead of a [V][frames] matrix: the sample can then be long enough
        oracle.bank_render(voices_desc, st, SR, FILTER_BIQUAD, frames, want_voices=False, want_bus=False,
                           nthreads=n_threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return voices_desc.shape[0] * frames / best, best


def cpu_baseline(args, bankgen):
    cores = os.cpu_count() or 1
    probe = bankgen.make_bank(max(cores * 4, 32), RENDER_FRAMES, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    rate, _ = cpu_port_throughput(probe, cores, 2048)
    want = max(rate * args.cpu_seconds, 1.0)
    nv = max(cores * 64, 1024)
    frames = int(min(max(want / nv // BLOCK, 1), 720)) * BLOCK      # at most one 60 s render per voice
    sample = bankgen.make_bank(nv, RENDER_FRAMES, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    rate, dt = cpu_port_throughput(sample, cores, frames)
    return {"value": rate, "unit": "voice-samples/s", "cores": cores, "kind": "port",
            "sample": f"{nv} voices x {frames} frames of the config-3 bank (biquad+ADSR), {dt:.1f} s, "
                      f"{cores} threads; C port of the reference's x16 path (Rust toolchain absent), gcc {_ORACLE_FLAGS}"}


# stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner to stdout at
# NCCL_DEBUG=VERSION), so file descriptor 1 points at stderr for the whole run and the result line goes to a
# saved copy of the original stdout.
_RESULT_FD = None


def capture_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (the C port: the Rust crate
    cannot be built in this image) on all host cores; each step is a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from synth2_b200 import bankgen     # numpy only: the product library (libs2cuda.so) is never loaded by this arm
    cores = os.cpu_count() or 1
    nv = max(cores * 64, 1024)          # enough voices per thread that thread start-up does not show (same as cpu_baseline)
    oracle = cpu_oracle()
    voices = bankgen.make_bank(nv, RENDER_FRAMES, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD,
                               pitches=oracle.pitch_table())
    st = oracle.bank_init_states(voices)
    frames = step_frames(args.steps, args.block)
    for _ in range(args.warmup):
        oracle.bank_render(voices, st, SR, FILTER_BIQUAD, args.block, want_voices=False, want_bus=False, nthreads=cores)
    st = oracle.bank_init_states(voices)
    t0 = time.perf_counter()
    for fr in frames:
        oracle.bank_render(voices, st, SR, FILTER_BIQUAD, fr, want_voices=False, want_bus=False, nthreads=cores)
    dt = time.perf_counter() - t0
    value = nv * sum(frames) / dt
    sample = (f"{nv} voices x {sum(frames)} frames of the config-3 bank per run, {cores} threads, C port of the reference "
              f"x16 path, gcc {_ORACLE_FLAGS}")
    emit({
        "impl": "reference", "metric": "voice-samples/sec (osc+biquad, 48 kHz)", "value": value,
        "unit": "voice-samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"config 3: osc + resonant biquad + ADSR, 48 kHz, 4096-frame blocks; CPU sample: {nv} voices of the "
                               f"65,536-voice bank over the same first {sum(frames)} frames from note-on",
                   "voices": nv, "block_frames": args.block, "render_frames": sum(frames)},
        "cpu_baseline": {"value": value, "unit": "voice-samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "voice-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


# ------------------------------------------------------------------------------------------
# parity of the timed render, and the other BASELINE configs

PARITY_VOICES = 64


def parity_of_timed_render(voices, final_state, last_block, frames, np):
    """The oracle (allowed here: the checker, after the timed region) renders PARITY_VOICES voices of the timed bank
    over the same frames from note-on; compared with the GPU: final oscillator phase and frame offset bit-for-bit,
    the last block's rows by max |err| (unscaled, and over the reference peak) and SNR."""
    oracle = cpu_oracle()
    V = voices.shape[0]
    total = sum(frames)
    # half spread evenly over the bank, half from the corner where the second-order low-pass is least
    # forgiving in binary32: the lowest cutoff x damping products among the voices whose cutoff follows the mod envelope
    even = np.linspace(0, V - 1, PARITY_VOICES // 2).astype(np.int64)
    corner_score = voices["lpf_freq_hz"].astype(np.float64) * voices["damping"] + np.where(voices["mod_env_to_lpf_freq"] != 0, 0.0, 1e9)
    corner = np.argsort(corner_score, kind="stable")[:PARITY_VOICES // 2]
    idx = np.unique(np.concatenate([even, corner]))
    sub = np.ascontiguousarray(voices[idx])
    st = oracle.bank_init_states(sub)
    t0 = time.perf_counter()
    if total > frames[-1]:
        oracle.bank_render(sub, st, SR, FILTER_BIQUAD, total - frames[-1], want_voices=False, want_bus=False,
                           nthreads=os.cpu_count() or 1)
    ref, _ = oracle.bank_render(sub, st, SR, FILTER_BIQUAD, frames[-1], want_bus=False, nthreads=os.cpu_count() or 1)
    dt = time.perf_counter() - t0
    got = last_block[idx.tolist(), :frames[-1]].cpu().numpy()
    err = np.abs(got.astype(np.float64) - ref.astype(np.float64))
    per_voice = err.max(axis=1)
    peak = float(np.max(np.abs(ref)))
    p_err, p_ref = float(np.sum(err * err)), float(np.sum(ref.astype(np.float64) ** 2))
    snr = float("inf") if p_err == 0.0 else 10.0 * float(np.log10(max(p_ref, 1e-300) / p_err))
    def sample(mask):
        e, r = err[mask], ref[mask].astype(np.float64)
        pe, pr = float(np.sum(e * e)), float(np.sum(r * r))
        return {"voices": int(mask.sum()), "max_abs_err": float(e.max()) if e.size else 0.0,
                "snr_db": float("inf") if pe == 0.0 else 10.0 * float(np.log10(max(pr, 1e-300) / pe))}
    in_corner = np.isin(idx, corner)
    gs = final_state[idx]
    over = [{"voice": int(idx[i]), "cutoff_hz": float(sub["lpf_freq_hz"][i]), "damping": float(sub["damping"][i]),
             "max_abs_err": float(per_voice[i])} for i in np.argsort(-per_voice)[:8] if per_voice[i] > 1e-4]
    return {"voices_checked": int(idx.size), "frames": int(total), "compared": f"last block ({frames[-1]} frames) and final state",
            "phase_bit_exact": bool(np.array_equal(gs["phase"].view(np.uint32), st["phase"].view(np.uint32))),
            "frame_offset_equal": bool(np.array_equal(gs["frame_offset"], st["frame_offset"])),
            "max_abs_err": float(per_voice.max()), "ref_peak": peak,
            "max_abs_err_over_ref_peak": float(per_voice.max()) / max(peak, 1e-30), "snr_db": snr,
            # the two halves of the sample apart: voices spread over the bank, and the low-cutoff x low-damping corner
            # where one ulp of cutoff moves the reference itself by several 1e-4 (DESIGN.md section 5)
            "spread_sample": sample(~in_corner), "corner_sample": sample(in_corner),
            "voices_over_1e-4_unscaled": over, "oracle_seconds": dt}


DUMP_SEED = 0
DUMP_MAX_FRAMES = 4 << 20           # of one row: 16 MiB
DUMP_ROW_BYTES = 40 << 20           # the sampled rows and their phases; the bus adds at most 16 MiB


def dump_outputs(out_dir, block, frames, final_state, bus, np, torch):
    """--dump-outputs: what a caller of the timed path holds after its last step, as float32 .npy files.
      last_block.npy  [n, frames]  that step's output rows: every voice when they fit in the budget, else the
                                   rows of n voices drawn with numpy's default_rng(DUMP_SEED), in voice order
      phase.npy       [n]          the oscillator phase the same voices carry out of the step
      bus.npy         [frames]     the step's part of the master bus (--master-bus only)
    The bank is a pure function of the arguments (bankgen is counter-based), so runs with the same arguments
    compare file for file."""
    V = block.shape[0]
    cols = min(frames, DUMP_MAX_FRAMES)
    n = min(V, max(1, DUMP_ROW_BYTES // (4 * (cols + 1))))
    idx = np.arange(V) if n == V else np.sort(np.random.default_rng(DUMP_SEED).choice(V, n, replace=False))
    rows = block.index_select(0, torch.as_tensor(idx, device=block.device))[:, :cols]
    out = {"last_block": rows.cpu().numpy(), "phase": final_state["phase"][idx]}
    if bus is not None:
        out["bus"] = bus[:cols].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def _timed(torch, stream, bank, body):
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    ev0.record(stream)
    body()
    bank.join(stream)
    ev1.record(stream)
    torch.cuda.synchronize()
    return ev0.elapsed_time(ev1) * 1e-3


def _peak_gbs():
    try:
        return float(json.loads((ROOT / "MEASURED_PEAKS.json").read_text())["hbm_gbs"])
    except Exception:
        return 6650.0


def _rate(voices, frames, seconds, **kw):
    vs = voices * frames / seconds
    return {"voices": voices, "frames_per_voice": frames, "seconds": seconds, "value": vs, "unit": "voice-samples/s",
            "roofline_frac": vs * BYTES_PER_VOICE_SAMPLE / 1e9 / _peak_gbs(), **kw}


def extra_config2(s2, bankgen, torch, stream, dev_index):
    """BASELINE config 2: 1,024 saw/square voices + one-pole low-pass, 4,096-frame buffers, time-split kernels.
    64 blocks from note-on (cutoff sweep + ramps), then 64 more (sustain); 16 rotating output buffers so a
    16 MiB block does not simply sit in the 126 MB L2."""
    V, T, blocks = 1024, 4096, 64
    voices = bankgen.make_bank(V, 4 * 2 * blocks * T)
    bank = s2.VoiceBank(voices, SR, s2.FILTER_ONE_POLE, device=dev_index, stream=stream)
    bank.set_time_split(True)
    ring = [torch.empty((V, T), device="cuda", dtype=torch.float32) for _ in range(16)]
    st = bank.get_state()
    for i in range(4):
        bank.render(T, ring[i & 15], T, None)
    bank.set_state(st)
    n0 = bank.time_split_blocks
    sec_a = _timed(torch, stream, bank, lambda: [bank.render(T, ring[i & 15], T, None) for i in range(blocks)])
    sec_b = _timed(torch, stream, bank, lambda: [bank.render(T, ring[i & 15], T, None) for i in range(blocks)])
    ts_blocks = bank.time_split_blocks - n0
    bank.close()
    return {"workload": "1,024 saw/square voices + one-pole low-pass, 48 kHz, 4,096-frame buffers, time-split kernels",
            "from_note_on": _rate(V, blocks * T, sec_a, blocks=blocks, us_per_block=sec_a / blocks * 1e6),
            "sustain": _rate(V, blocks * T, sec_b, blocks=blocks, us_per_block=sec_b / blocks * 1e6),
            "time_split_blocks": int(ts_blocks)}


def extra_config5(s2, bankgen, torch, stream, dev_index, seconds=2):
    """BASELINE config 5, one GPU's share: 32,768 patch variants (32 cutoffs x 32 dampings x 32 detunes of the default
    patch, second-order low-pass), every variant's render kept on the device; the first `seconds` s from note-on."""
    V, total, T = bankgen.SWEEP_VARIANTS, seconds * SR, BLOCK
    voices = bankgen.make_sweep_bank(0, 10 * SR)
    bank = s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, device=dev_index, stream=stream)
    bank.set_pipeline(4)
    out = torch.empty((V, total), device="cuda", dtype=torch.float32)
    st = bank.get_state()
    for i in range(3):
        bank.render(T, out[:, i * T:], total, None)
    bank.set_state(st)

    def body():
        pos = 0
        while pos < total:
            fr = min(T, total - pos)
            bank.render(fr, out[:, pos:], total, None)
            pos += fr
    sec = _timed(torch, stream, bank, body)
    finite = bool(torch.isfinite(out[:, -T:]).all())
    bank.close()
    del out
    torch.cuda.empty_cache()
    return {"workload": f"32,768 patch variants (cutoff x resonance x detune grid of the default patch), biquad, first {seconds} s "
                        f"from note-on, renders kept on the device ({V * total * 4 / 1e9:.1f} GB)",
            **_rate(V, total, sec, all_finite=finite)}


def extra_config4(s2, bankgen, torch, dist, stream, rank, world, dev_index, rank_max, barrier, seconds=2):
    """BASELINE config 4: a 262,144-voice bank sharded over the N GPUs as contiguous voice ranges; every rank renders
    its rows and its share of the master bus (in-kernel mix), then ONE NCCL reduce (s2_bank_reduce_bus) sums the
    whole-render buses into rank 0's master buffer.  Three timed passes give the breakdown: rows only, rows + mix,
    rows + mix + reduce (all inside the timed region of the third)."""
    from synth2_b200.shard import MasterBus, voice_range
    lo, hi = voice_range(rank, world, 262144)
    V, T = hi - lo, BLOCK
    blocks = (seconds * SR + T - 1) // T
    total = blocks * T
    voices = bankgen.make_bank(V, 10 * SR, first_voice=lo, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    bank = s2.VoiceBank(voices, SR, s2.FILTER_BIQUAD_LP, device=dev_index, stream=stream)
    bank.set_pipeline(4)
    ring = [torch.empty((V, T), device="cuda", dtype=torch.float32) for _ in range(2)]
    bus = torch.zeros(total, device="cuda", dtype=torch.float32)
    master = torch.zeros(total, device="cuda", dtype=torch.float32)
    comm = MasterBus(rank, world, dev_index)
    st = bank.get_state()
    for i in range(3):
        bank.render(T, ring[i & 1], T, bus[:T])
    comm.reduce(bank, bus, master, root=0, stream=stream)       # warm the communicator up

    def run(mix, reduce):
        bank.set_state(st)
        barrier()
        ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        ev0.record(stream)
        for i in range(blocks):
            bank.render(T, ring[i & 1], T, bus[i * T:(i + 1) * T] if mix else None)
        bank.join(stream)
        ev1.record(stream)
        if reduce:
            comm.reduce(bank, bus, master, root=0, stream=stream)
        ev2.record(stream)
        barrier()
        return rank_max(ev0.elapsed_time(ev2)) * 1e-3, rank_max(ev1.elapsed_time(ev2)) * 1e-3

    t_rows, _ = run(False, False)
    t_mix, _ = run(True, False)
    t_all, t_reduce = run(True, True)
    finite = bool(torch.isfinite(master).all()) if rank == 0 else True
    comm.close()
    bank.close()
    vs = 262144 * total / t_all
    return {"workload": f"262,144 voices over {world} GPUs ({V} per GPU, contiguous ranges), osc + biquad + ADSR, first {seconds} s "
                        "from note-on; per-voice rows + in-kernel mono mix per block, then one NCCL reduce of the whole-render bus "
                        "(s2_bank_reduce_bus) inside the timed region",
            "value": vs, "unit": "voice-samples/s", "roofline_frac_per_gpu": vs / world * BYTES_PER_VOICE_SAMPLE / 1e9 / _peak_gbs(),
            "blocks": blocks, "us_per_block": {"render_rows_only": t_rows / blocks * 1e6, "mix_added": (t_mix - t_rows) / blocks * 1e6,
                                               "total": t_all / blocks * 1e6},
            "reduce_us_total": t_reduce * 1e6, "reduce_bytes": total * 4, "master_bus": "mono (the reference mixes to one "
            "channel and its player copies it to both, audio_player.rs:136-199)", "all_finite": finite}


def main():
    sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written or cached there
    args = parse()
    capture_stdout()
    if args.impl == "reference":
        run_reference(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import synth2_b200 as s2
    from synth2_b200 import bankgen

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the renderer has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    V, T = args.voices, args.block
    frames = step_frames(args.steps, T)
    total_frames = sum(frames)
    voices = bankgen.make_bank(V, RENDER_FRAMES, first_voice=rank * V, mod_to_lpf_choices=bankgen.MOD_TO_LPF_BIQUAD)
    stream = torch.cuda.current_stream()
    bank = s2.VoiceBank(voices, SR, FILTER_BIQUAD, device=local, stream=stream)
    if args.pipeline > 1:
        bank.set_pipeline(args.pipeline)
    ring = [torch.empty((V, T), device=dev, dtype=torch.float32) for _ in range(2)]   # 2 x 1 GiB
    state0 = bank.get_state()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def rank_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- value: device-resident render ------------------------------------------------------
    want_master = args.master_bus and world > 1
    master = torch.zeros(total_frames, device=dev, dtype=torch.float32) if want_master else None
    for i in range(max(args.warmup, 3)):
        bank.render(T, ring[i & 1], T, None)
    bank.set_state(state0)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    step_ev = [torch.cuda.Event(enable_timing=True) for _ in frames]
    launches0 = s2.lib().s2_launch_count()
    clocks = ClockSampler(local)
    with clocks:
        ev0.record(stream)
        pos = 0
        for i, fr in enumerate(frames):
            bank.render(fr, ring[i & 1], T, master[pos:pos + fr] if want_master else None)
            pos += fr
            bank.join(stream)        # pipelined banks: the timing stream waits for every voice range of this step
            step_ev[i].record(stream)
        if want_master:
            dist.reduce(master, dst=0, op=dist.ReduceOp.SUM)
        ev1.record(stream)
        barrier()
    launches = s2.lib().s2_launch_count() - launches0
    ms = rank_max(ev0.elapsed_time(ev1))
    value = world * V * total_frames / (ms * 1e-3)
    step_ms = [(ev0 if i == 0 else step_ev[i - 1]).elapsed_time(step_ev[i]) for i in range(len(frames))]
    final_state = bank.get_state()
    assert np.all(final_state["frame_offset"] == total_frames)
    assert bool(torch.isfinite(ring[(len(frames) - 1) & 1][:, :frames[-1]]).all())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ring[(len(frames) - 1) & 1], frames[-1], final_state,
                     master[total_frames - frames[-1]:] if want_master else None, np, torch)

    # ---- parity of the timed render against the CPU oracle (after the timed region) -------------
    parity = None
    if rank == 0 and not args.no_parity:
        parity = parity_of_timed_render(voices, final_state, ring[(len(frames) - 1) & 1], frames, np)

    # ---- clocks: an NVML query takes milliseconds, so a 6 ms timed region yields one sample.  Repeat the same
    # render untimed, right away, under the sampler until there are a few (the e2e pass below is left alone: a
    # sampling thread next to its host loop costs it 5-20 %)
    timed_samples = len(clocks.samples)
    repeats = 0
    while clocks._nv and len(clocks.samples) < 8 and repeats < 16:
        bank.set_state(state0)
        with clocks:
            for i, fr in enumerate(frames):
                bank.render(fr, ring[i & 1], T, None)
            bank.join(stream)
            torch.cuda.synchronize()
        repeats += 1

    # ---- e2e: host-buffer calls, H2D + D2H inside the timed region ----------------------------
    e2e = None
    if not args.no_e2e:
        rel_host = torch.from_numpy(voices["release_offset"].astype(np.uint32).view(np.int32)).pin_memory()
        bus_host = [torch.empty(T, dtype=torch.float32).pin_memory() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        checksum = 0.0

        def e2e_pass(n_steps_frames):
            """Two buffers in flight, like the reference's player (audio_player.rs:56-60): enqueue step i,
            then wait for and consume step i-1."""
            nonlocal checksum
            for i, fr in enumerate(n_steps_frames):
                bank.set_releases(rel_host)                                              # H2D, pinned
                bank.render_bus_host_async(fr, bus_host[i & 1], ring[i & 1], T)          # render + mix + D2H
                done[i & 1].record(stream)
                if i > 0:
                    done[(i - 1) & 1].synchronize()
                    checksum += float(bus_host[(i - 1) & 1][0])                          # the host reads the result
            done[(len(n_steps_frames) - 1) & 1].synchronize()
            checksum += float(bus_host[(len(n_steps_frames) - 1) & 1][0])

        bank.set_state(state0)
        e2e_pass([T] * 3)
        bank.set_state(state0)
        barrier()
        t0 = time.perf_counter()
        ev0.record(stream)
        e2e_pass(frames)
        bank.join(stream)
        ev1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        assert np.isfinite(checksum)
        e_ms = rank_max(max(ev0.elapsed_time(ev1), wall * 1e3))
        e2e = {"value": world * V * total_frames / (e_ms * 1e-3), "unit": "voice-samples/s",
               "h2d_bytes_per_step": int(rel_host.numel() * 4), "d2h_bytes_per_step": int(T * 4),
               "ms_per_step": e_ms / len(frames),
               "what": "per step: note-off table H2D (pinned), render into the device ring + mono mix, mix D2H to "
                       "pinned host (the Synth::sample result), host waits for and reads the previous step's mix "
                       "(two buffers in flight, as the reference's audio_player does); wall clock"}
    bank.close()
    del ring, bank
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs --------------------------------------------------------------
    extra = None
    if not args.no_extra:
        extra = {}
        if world == 1:
            extra["config2"] = extra_config2(s2, bankgen, torch, stream, local)
            extra["config5"] = extra_config5(s2, bankgen, torch, stream, local)
        else:
            extra["config4"] = extra_config4(s2, bankgen, torch, dist, stream, rank, world, local, rank_max, barrier)

    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    n_ranges = max(int(args.pipeline), 1)
    per_launch_bytes = V * T * BYTES_PER_VOICE_SAMPLE // n_ranges
    achieved = V * total_frames * BYTES_PER_VOICE_SAMPLE / (ms * 1e-3) / 1e9
    # a step is `n_ranges` launches of the render kernel (one per voice range, on internal streams: they overlap
    # with each other and with the neighbouring steps), so the per-launch duration that matters is the step's
    # share: step time / launches per step
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "kernel": "s2::render_kernel<FILTER=biquad low-pass, TRACE=0>: one voice per lane, one warp per block",
                "peak_source": peak_src, "launches_per_step": n_ranges, "algorithmic_bytes_per_launch": per_launch_bytes,
                "algorithmic_bytes_per_step": V * T * BYTES_PER_VOICE_SAMPLE,
                "avg_step_ms": ms / len(frames), "avg_launch_ms": ms / len(frames) / n_ranges,
                "avg_launch_ms_note": "launches of one step overlap (4 streams): step time / launches per step, not the "
                                      "serialised duration ncu reports for a launch running alone"}
    prof = ROOT / "profiles" / "traffic.json"
    if prof.exists():
        try:
            roofline["traffic"] = json.loads(prof.read_text()).get("render_kernel_bytes_per_launch")
        except Exception:
            pass

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args, bankgen)

    if rank == 0:
        emit({
            "metric": "voice-samples/sec (osc+biquad, 48 kHz)", "value": value, "unit": "voice-samples/s",
            "n_gpus": world, "steps": len(frames), "warmup": max(args.warmup, 3), "ms_per_step": ms / len(frames),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config 3: 65,536 voices/GPU, osc (saw/square) + resonant biquad + ADSR, 48 kHz, 4,096-frame "
                                   f"blocks, state carried on device; this run renders frames [0, {total_frames}) of the 60 s render "
                                   f"= the first {total_frames / SR:.2f} s after note-on"
                                   + (" (the whole render)" if total_frames == RENDER_FRAMES else
                                      " (cutoff sweep for 0.2 s, then attack / decay ramps for up to 1 s, then sustain)"),
                       "voices_per_gpu": V, "block_frames": T, "render_frames": total_frames,
                       "l2_hygiene": "each step writes a fresh 1 GiB block (ring of 2) >> 126 MB L2; no input is re-read",
                       "master_bus": bool(want_master), "pipeline_voice_ranges": int(args.pipeline)},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "launches_per_step": launches / len(frames),
            "clocks": {**clocks.summary(), "samples_in_timed_region": timed_samples, "untimed_repeats_sampled": repeats}, "step_ms": [round(x, 4) for x in step_ms], "parity": parity, "extra": extra,
        })
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
