"""References for the mono bus (`d_bus_out` of s2_bank_render): exact-sum voice banks with their closed form, and
the error bound of the bus's summation trees.  Shared by test_gpu_bus.py and test_gpu_parity.py."""
import math

import numpy as np

from synth2_b200._lib import NO_RELEASE, OSC_SQUARE, VOICE_DESC

U = 2.0 ** -24          # unit roundoff of binary32
GRID = 2.0 ** -14       # every sample of an exact bank is an integer multiple of this
TILE_FRAMES = 64        # kTileFrames (s2_internal.h): frames per write-back tile of the render kernel
BUS_COUNTERS = 1024     # kBusCounters (s2_internal.h): frame groups of 128 the wide reduction can count


def exact_bank(n, seed, tail_safe=False, span=40000):
    """n one-pole voices whose every output sample is +-c_i * 2^-14 or 0, with integer c_i in [1, 255].

    - lpf_freq_hz = 1e9: k = exp(-2 pi f / sr) = 0 at any mod-envelope amount, so the filter passes y = u exactly;
    - osc_gain = +-2^26: the x16 path adds the gain (process.rs:341-345) and RN(RN(osc + G) + RN(nz + amt)) = G,
      since |osc| <= 1 and |nz + amt| <= 2 are below half an ulp of 2^26 (4);
    - amp_sustain = c_i * 2^-40 and frame_offset past attack + decay: a sounding frame is G * sustain exactly;
    - amp_release_ms = 0: the sample is 0 from the release offset on.
    Random kinds, seeds, pitches (30-5000 Hz), noise amounts {0, 0.5, 1}, offsets, note-offs within `span` frames
    of the start (some voices held, some released before it), mod->cutoff amounts {0, 10, -3} with the mod
    envelope in its decay, and 10 % inactive voices.  Attack and decay lengths differ, so banks wider than a warp
    are permuted into slots.  So long as sum(c_i) < 2^24 every partial sum is exact and the float32 bus equals the
    float64 sum of the rows in any summation order.

    tail_safe: square oscillators and no noise, for calls whose `frames % 16` tail frames take the scalar path
    (sample = osc * G + nz * amt): there a sounding sample is +-c_i * 2^-14 with the square wave's sign."""
    rng = np.random.default_rng(seed)
    b = np.zeros(n, dtype=VOICE_DESC)
    b["osc_kind"] = OSC_SQUARE if tail_safe else rng.integers(0, 4, n)
    b["noise_seed"] = rng.integers(0, 1 << 32, n, dtype=np.uint64).astype(np.uint32)
    b["pitch_hz"] = np.exp(rng.uniform(np.log(30.0), np.log(5000.0), n)).astype(np.float32)
    b["osc_gain"] = np.where(rng.random(n) < 0.5, -1.0, 1.0) * 2.0 ** 26
    b["noise_amt"] = 0.0 if tail_safe else rng.choice([0.0, 0.5, 1.0], n)
    b["lpf_freq_hz"] = 1e9
    b["damping"] = 1.0
    b["amp_attack_ms"] = rng.uniform(0.0, 20.0, n)
    b["amp_decay_ms"] = rng.uniform(0.0, 20.0, n)
    b["amp_sustain"] = rng.integers(1, 256, n) * 2.0 ** -40
    b["amp_release_ms"] = 0.0
    b["mod_attack_ms"] = 0.0
    b["mod_decay_ms"] = rng.uniform(500.0, 5000.0, n)
    b["mod_sustain"] = rng.uniform(0.0, 1.0, n)
    b["mod_env_to_lpf_freq"] = rng.choice([0.0, 10.0, -3.0], n)
    b["frame_offset"] = 2000 + rng.integers(0, 30000, n)          # past attack + decay (<= 1,920 frames)
    rel = b["frame_offset"].astype(np.int64) + rng.integers(-500, span, n)
    b["release_offset"] = np.where(rng.random(n) < 0.3, NO_RELEASE, np.maximum(rel, 0)).astype(np.uint32)
    b["active"] = rng.random(n) < 0.9
    return b


def closed_form(voices, n0, frames, release=None):
    """Rows of an exact bank for one x16-only call starting at per-voice frame offsets n0: row i is val[i] for
    the first stop[i] frames and 0 after.  val = sign(G) * c * 2^-14 for active voices; a frame n sounds while
    (float)n < (float)release (all offsets here are below 2^24, so that is n < release)."""
    active = voices["active"] != 0
    val = (np.sign(voices["osc_gain"]) * voices["amp_sustain"].astype(np.float64) * 2.0 ** 26).astype(np.float32)
    rel = (voices["release_offset"] if release is None else np.asarray(release)).astype(np.int64)
    stop = np.clip(rel - np.asarray(n0, dtype=np.int64), 0, frames)
    val[~active] = 0.0
    stop[~active] = 0
    return val, stop


def advance(voices, n0, frames):
    """Frame offsets after a call of `frames` frames (inactive voices do not move)."""
    return np.asarray(n0, dtype=np.int64) + np.where(voices["active"] != 0, int(frames), 0)


def closed_bus(val, stop, frames):
    """The exact bus of closed-form rows, as binary32 with +0.0 for silence."""
    d = np.zeros(int(frames) + 1, dtype=np.float64)
    np.add.at(d, stop, -val.astype(np.float64))
    d[0] += float(np.sum(val, dtype=np.float64))
    return (np.cumsum(d[:-1]) + 0.0).astype(np.float32)


def closed_rows(val, stop, frames):
    return np.where(np.arange(frames)[None, :] < stop[:, None], val[:, None], np.float32(0.0))


def reference_order_bus(rows):
    """synth.rs:176-202: acc = 0.0; acc += row[v] for v in voice order, in binary32."""
    acc = np.zeros(rows.shape[1], dtype=np.float32)
    for r in rows:
        acc = acc + r.astype(np.float32)
    return acc


def bus_depth(n_voices, frames, path):
    """Depth d of the summation tree that makes the bus of one call: the most roundings on any row's way to it.

    In-warp partial (render kernel, one warp = 32 slots):
      a full 64-frame tile (frames % 4 == 0): each lane adds its 16 rows as two pairwise 8-row trees (3 levels),
        adds the two (1), then the butterfly shuffle adds the other q-group (1): 5;
      a ragged tile (the last one when frames % 64 != 0; all of them when frames % 4 != 0): four accumulators of
        8 rows each from 0.0 (8), then ((a0 + a1) + (a2 + a3)) (2): 10.
    Reduction over R partial rows:
      narrow (bus_reduce_kernel): 8 warps take every 8th row, 4 rotating accumulators: ceil(R/32) adds, then
        2 levels over the accumulators and 7 sequential adds over the 8 warps: ceil(R/32) + 9;
      wide (bus_reduce_wide_kernel, R >= 512, frames % 128 == 0 and frames / 128 <= kBusCounters): 4 quarters of
        the rows, 8 warps each, 2 accumulators: ceil(R/64) adds, 1 to join them, 7 over the warps, 3 over the
        quarters: ceil(R/64) + 11.
    R is the number of warps on the default and pipelined paths (their partial rows), the number of voices on the
    time-split path (its output rows, reduced by the narrow kernel).  Banks of <= 32 voices sum in voice order:
    d = n_voices."""
    if n_voices <= 32:
        return n_voices
    if path == "time_split":
        return math.ceil(n_voices / 32) + 9
    warps = math.ceil(n_voices / 32)
    in_warp = 5 if frames % 4 == 0 and frames % TILE_FRAMES == 0 else 10
    wide = warps >= 512 and frames % 128 == 0 and frames // 128 <= BUS_COUNTERS
    return in_warp + (math.ceil(warps / 64) + 11 if wide else math.ceil(warps / 32) + 9)


def assert_bus_within_bound(bus, rows, n_voices, path, what=""):
    """|bus - sum_f64(rows)| <= gamma_d * sum|rows| frame by frame, gamma_d = d u / (1 - d u) (the classic bound
    of recursive summation, applied along each row's path through the tree; d from bus_depth).  `rows` are the
    rows the same render produced ([V, frames] numpy or torch, any float type)."""
    if hasattr(rows, "double"):
        exact = rows.double().sum(dim=0).cpu().numpy()
        mag = rows.double().abs().sum(dim=0).cpu().numpy()
    else:
        exact = rows.astype(np.float64).sum(axis=0)
        mag = np.abs(rows.astype(np.float64)).sum(axis=0)
    bus = np.asarray(bus.cpu().numpy() if hasattr(bus, "cpu") else bus, dtype=np.float64)
    assert bus.shape == exact.shape and np.all(np.isfinite(bus)), what
    d = bus_depth(n_voices, bus.shape[0], path)
    gamma = d * U / (1.0 - d * U)
    err = np.abs(bus - exact)
    worst = int(np.argmax(err - gamma * mag))
    assert np.all(err <= gamma * mag), (f"{what}: |bus - sum| = {err[worst]:.3e} at frame {worst} exceeds "
                                        f"gamma_{d} * sum|rows| = {gamma * mag[worst]:.3e}")
