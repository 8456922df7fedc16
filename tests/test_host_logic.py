"""CPU-only checks of the host side: the C ABI library loads and exports exactly what
include/s2_cuda.h declares, struct layouts agree across header / ctypes / oracle, the host helpers
match the oracle, and the library refuses to compute without a GPU (no CPU fallback)."""
import ctypes as C
import pathlib
import re
import subprocess

import numpy as np
import pytest

import oracle
import synth2_b200 as s2
from synth2_b200 import _lib, bankgen
from synth2_b200.shard import voice_range

ROOT = pathlib.Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "s2_cuda.h").read_text()


def declared_functions():
    body = re.sub(r"/\*.*?\*/", "", HEADER, flags=re.S)
    return sorted(set(re.findall(r"\b(s2_[a-z0-9_]+)\s*\(", body)))


def test_library_exports_every_declared_symbol():
    names = declared_functions()
    assert len(names) >= 20
    handle = C.CDLL(str(_lib.LIB_PATH))
    for n in names:
        assert hasattr(handle, n), f"{n} declared in s2_cuda.h but not exported"
    assert sorted(_lib.SYMBOLS) == names, "ctypes table and header disagree"


def test_abi_version_and_error_string():
    assert s2.lib().s2_abi_version() == 1
    assert isinstance(s2.lib().s2_last_error(), bytes)


def _c_struct_fields(name):
    m = re.search(r"typedef struct " + name + r" \{(.*?)\} " + name + ";", HEADER, re.S)
    body = re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, rest = decl.split(None, 1)
        for f in rest.split(","):
            fields.append((f.strip(), ctype))
    return fields


@pytest.mark.parametrize("cname,dtype", [("s2_voice_desc", s2.VOICE_DESC), ("s2_voice_state", s2.VOICE_STATE)])
def test_struct_layout_matches_header(cname, dtype):
    fields = _c_struct_fields(cname)
    assert [f for f, _ in fields] == list(dtype.names)
    for (f, ctype), n in zip(fields, dtype.names):
        want = {"uint32_t": "<u4", "float": "<f4"}[ctype]
        assert dtype[n].str == want, f
    assert dtype.itemsize == 4 * len(fields)


def test_oracle_voice_desc_has_the_same_layout():
    src = (ROOT / "oracle" / "s2_oracle.h").read_text()
    m = re.search(r"typedef struct \{([^}]*)\} s2o_voice_desc;", src, re.S)
    body = re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [f.strip() for f in decl.split(None, 1)[1].split(",")]
    assert names == list(s2.VOICE_DESC.names)
    m = re.search(r"typedef struct \{([^}]*)\} s2o_voice_state;", src, re.S)
    body = re.sub(r"/\*.*?\*/", "", m.group(1), flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            names += [f.strip() for f in decl.split(None, 1)[1].split(",")]
    assert names == list(s2.VOICE_STATE.names)


def test_note_to_pitch_matches_oracle_for_all_notes():
    for n in range(128):
        a = np.float32(s2.note_to_pitch(n))
        b = np.float32(oracle.lib().s2o_note_to_pitch(n))
        assert a.tobytes() == b.tobytes()
    assert s2.note_to_pitch(69) == 440.0


def test_default_voice_is_the_reference_default_patch():
    d = s2.default_voice(1)[0]
    cfg = oracle.default_config()[0]
    assert d["osc_kind"] == cfg["osc_kind"] == s2.OSC_SAW
    assert d["osc_gain"] == cfg["osc_gain"] == 1.0
    assert d["noise_amt"] == cfg["noise"] == 0.0
    assert d["lpf_freq_hz"] == cfg["lpf_freq"] == 200.0
    assert (d["amp_attack_ms"], d["amp_decay_ms"], d["amp_sustain"], d["amp_release_ms"]) == (100.0, 100.0, 0.5, 100.0)
    assert tuple(cfg["amp_env"]) == (100.0, 100.0, 0.5, 100.0)
    assert (d["mod_attack_ms"], d["mod_decay_ms"], d["mod_sustain"], d["mod_release_ms"]) == (0.0, 200.0, 0.0, 0.0)
    assert tuple(cfg["mod_env"]) == (0.0, 200.0, 0.0, 0.0)
    assert d["mod_env_to_osc_freq"] == cfg["mod_env_to_osc_freq"] == 0.0
    assert d["mod_env_to_lpf_freq"] == cfg["mod_env_to_lpf_freq"] == 10.0
    assert d["release_offset"] == s2.NO_RELEASE and d["active"] == 0


def test_no_cpu_fallback():
    """Without a GPU every compute entry must fail loudly; with one, this test is a no-op."""
    n = C.c_int(0)
    rc = s2.lib().s2_device_count(C.byref(n))
    if rc == 0 and n.value > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(s2.S2Error) as e:
        s2.VoiceBank(bankgen.make_bank(4, 64), 48000, 0)
    assert e.value.code == _lib.S2_ERR_NO_DEVICE
    with pytest.raises(s2.S2Error):
        s2.Synth()


def test_argument_validation_happens_before_the_device():
    h = C.c_void_p()
    v = bankgen.make_bank(2, 64)
    rc = s2.lib().s2_bank_create(0, 48000, 0, 0, _lib.ptr(v), None, C.byref(h))
    assert rc == _lib.S2_ERR_INVALID
    rc = s2.lib().s2_bank_create(0, 0, 0, 2, _lib.ptr(v), None, C.byref(h))
    assert rc == _lib.S2_ERR_INVALID
    rc = s2.lib().s2_bank_create(0, 48000, 6, 2, _lib.ptr(v), None, C.byref(h))      # kinds 0..5 exist
    assert rc == _lib.S2_ERR_INVALID
    assert b"filter_kind" in s2.lib().s2_last_error()
    assert s2.lib().s2_bank_render(None, 16, None, 0, None) == _lib.S2_ERR_INVALID
    assert s2.lib().s2_synth_note_on(None, 60, 1.0) == _lib.S2_ERR_INVALID


def test_product_code_never_touches_the_oracle():
    for p in list((ROOT / "synth2_b200").rglob("*.py")) + list((ROOT / "synth2_b200" / "csrc").glob("*.cu")) \
            + list((ROOT / "synth2_b200" / "csrc").glob("*.h")):
        text = p.read_text()
        assert "s2o_" not in text and "libs2oracle" not in text and "import oracle" not in text, p


# ---- synthetic bank generator --------------------------------------------------------------

def test_bankgen_is_counter_based():
    whole = bankgen.make_bank(100, 48000)
    part = bankgen.make_bank(40, 48000, first_voice=60)
    assert whole[60:].tobytes() == part.tobytes()
    assert whole["release_offset"][0] == 36000 and 36000 % 16 == 0
    assert np.all((whole["lpf_freq_hz"] >= 100) & (whole["lpf_freq_hz"] <= 8000))
    assert np.all((whole["damping"] >= 0.2) & (whole["damping"] <= 1.4141))
    assert set(np.unique(whole["mod_env_to_lpf_freq"])) <= {0.0, 10.0}
    assert np.all(whole["noise_seed"] == np.arange(100))
    assert list(whole["osc_kind"][:4]) == [s2.OSC_SAW, s2.OSC_SQUARE, s2.OSC_SAW, s2.OSC_SQUARE]


def test_sweep_bank_is_the_config5_grid():
    """BASELINE config 5: 32 cutoffs x 32 dampings x 32 detunes per GPU, MIDI note 48 + 4 * gpu."""
    cutoff, damping, cents = bankgen.sweep_axes()
    assert cutoff[0] == np.float32(100.0) and cutoff[-1] == np.float32(12800.0)
    assert np.allclose(np.diff(np.log2(cutoff.astype(np.float64))), 7.0 / 31.0, atol=1e-6)
    assert damping[0] == np.float32(0.2) and damping[-1] == np.float32(1.414)
    assert cents[0] == -50.0 and cents[-1] == 50.0
    b = bankgen.make_sweep_bank(2, 480000)
    assert b.shape == (32768,) and np.all(b["active"] == 1)
    # variant id = (cutoff * 32 + damping) * 32 + detune
    vid = (7 * 32 + 19) * 32 + 3
    assert b["lpf_freq_hz"][vid] == cutoff[7] and b["damping"][vid] == damping[19]
    base = float(np.float32(s2.note_to_pitch(48 + 8)))
    assert b["pitch_hz"][vid] == np.float32(base * 2.0 ** (cents[3] / 1200.0))
    assert len(np.unique(b[["pitch_hz", "lpf_freq_hz", "damping"]])) == 32768          # all variants distinct
    # the mod envelope never opens the cutoff beyond 0.45 * sr (the biquad is unstable above Nyquist)
    peak = b["lpf_freq_hz"].astype(np.float64) * np.exp2(b["mod_env_to_lpf_freq"].astype(np.float64))
    assert peak.max() <= 0.45 * 48000 * (1 + 1e-6) and b["mod_env_to_lpf_freq"].min() >= 0.0
    assert b["release_offset"][0] == 360000
    # any slice of the grid can be generated on its own (ranks / chunks)
    part = bankgen.make_sweep_bank(2, 480000, first_variant=1000, n_variants=77)
    assert part.tobytes() == b[1000:1077].tobytes()
    # the rest is the default patch
    d = s2.default_voice(1)[0]
    for f in ("amp_attack_ms", "amp_decay_ms", "amp_sustain", "amp_release_ms", "mod_decay_ms", "osc_gain", "noise_amt"):
        assert np.all(b[f] == d[f]), f
    with pytest.raises(ValueError):
        bankgen.make_sweep_bank(0, 480000, first_variant=32768, n_variants=1)


def test_sweep_banks_of_different_gpus_differ_only_in_the_note():
    """Config 5 shards by GPU index with no exchange: rank g renders the same 32 x 32 x 32 grid at note 48 + 4 g."""
    a, b = bankgen.make_sweep_bank(0, 480000, n_variants=2048), bankgen.make_sweep_bank(3, 480000, n_variants=2048)
    for f in a.dtype.names:
        if f == "pitch_hz":
            ratio = b[f].astype(np.float64) / a[f].astype(np.float64)
            assert np.allclose(ratio, 2.0 ** (12 / 12.0), rtol=1e-6)          # 3 GPUs x 4 semitones = one octave
        else:
            assert np.array_equal(a[f], b[f]), f
    with pytest.raises(ValueError):
        bankgen.make_sweep_bank(20, 480000)                                  # note 128 does not exist


def test_splitmix64_known_answer():
    # splitmix64 reference stream for seed 0: first output
    assert int(bankgen.splitmix64(np.array([0], dtype=np.uint64))[0]) == 0xE220A8397B1DCDAF


# ---- sharding --------------------------------------------------------------------------------

@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_voice_ranges_partition(world):
    n = 262144 + 5
    spans = [voice_range(r, world, n) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    for a, b in zip(spans[:-1], spans[1:]):
        assert a[1] == b[0]
    sizes = [b - a for a, b in spans]
    assert max(sizes) - min(sizes) <= 1


def _shard_worker(rank, world, port, q):
    import os
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from synth2_b200.shard import reduce_master_bus
    V, T = 48, 512
    lo, hi = voice_range(rank, world, V)
    mine = bankgen.make_bank(hi - lo, 4 * T, first_voice=lo, kinds=(0, 1, 2, 3))
    st = oracle.bank_init_states(mine)
    _, bus = oracle.bank_render(mine, st, 48000, 0, T)         # CPU stand-in for the per-GPU render
    t = torch.from_numpy(bus.copy())
    reduce_master_bus(t, dst=0)
    if rank == 0:
        q.put(t.numpy().copy())
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_master_bus_world2_gloo():
    """N>1 path on CPU: each rank renders its voice range, one reduce sums the buses on rank 0."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    V, T = 48, 512
    full = bankgen.make_bank(V, 4 * T, kinds=(0, 1, 2, 3))
    st = oracle.bank_init_states(full)
    _, want = oracle.bank_render(full, st, 48000, 0, T)
    np.testing.assert_allclose(got, want, atol=1e-4 * max(1.0, float(np.max(np.abs(want)))), rtol=0)


def test_bench_reference_arm_runs_on_cpu():
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0


def test_bench_dump_outputs_is_a_fixed_sample_within_64_mib(tmp_path):
    """bench.py --dump-outputs: a 65,536-voice block is sampled to the same voices on every call and stays under
    64 MiB; a narrow block is written whole; the rows, their phases and the bus are float32."""
    import torch
    import bench
    for V, T, bus in ((65536, 4096, None), (300, 1000, torch.linspace(-1, 1, 1000))):
        block = torch.arange(V, dtype=torch.float32)[:, None].expand(V, T)      # row v holds v
        st = np.zeros(V, dtype=s2.VOICE_STATE)
        st["phase"] = np.arange(V, dtype=np.float32)
        dirs = [tmp_path / f"{V}_a", tmp_path / f"{V}_b"]
        for d in dirs:
            bench.dump_outputs(str(d), block, T, st, bus, np, torch)
        files = sorted(p.name for p in dirs[0].iterdir())
        assert files == (["bus.npy", "last_block.npy", "phase.npy"] if bus is not None else ["last_block.npy", "phase.npy"])
        assert sum(p.stat().st_size for p in dirs[0].iterdir()) <= 64 << 20
        rows, phase = np.load(dirs[0] / "last_block.npy"), np.load(dirs[0] / "phase.npy")
        assert rows.dtype == phase.dtype == np.float32 and rows.shape == (phase.size, T)
        assert np.array_equal(rows[:, 0], phase) and np.all(rows == rows[:, :1])      # each row beside its phase
        assert np.all(np.diff(phase) > 0)
        assert phase.size == min(V, bench.DUMP_ROW_BYTES // (4 * (T + 1)))
        if bus is not None:
            assert np.load(dirs[0] / "bus.npy").tobytes() == bus.numpy().tobytes()
        for name in files:
            assert (dirs[0] / name).read_bytes() == (dirs[1] / name).read_bytes()


def test_math_kernels_round_once_on_cpu(tmp_path):
    """synth2_b200/csrc/s2_math.h (2^x, e^x, sin/cos used for filter coefficients) is host-and-device code:
    compiled for the CPU it must return the once-rounded binary64 result on dense sweeps (tools/check_math.cpp)."""
    import shutil
    import subprocess
    if shutil.which("g++") is None:
        pytest.skip("no g++")
    exe = tmp_path / "check_math"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-march=x86-64-v3", "-o", str(exe),
                    str(ROOT / "tools" / "check_math.cpp")], check=True, capture_output=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout
    assert "special values ok" in out.stdout


# ---- .synth2 patch files (csrc/s2_patch.cpp; runs without a GPU) -------------------------------

from synth2_b200 import patch as s2patch

EXAMPLE_SYNTH2 = "synth mySynth {\n\n}\n"          # the reference's example.synth2, verbatim


def test_moving_cutoff_functions_on_cpu(tmp_path):
    """synth2_b200/csrc/s2_cutoff.h compiles for the CPU: the straight-line division, e^-theta, the windowed
    sin / cos, the division by the sample rate (every numerator at the usual rates), 2^x around a window centre and
    a whole decay sweep at the worst corner against the full evaluation (tools/check_cutoff.cpp)."""
    import shutil
    import subprocess
    if not shutil.which("g++"):
        pytest.skip("g++ not available")
    exe = tmp_path / "check_cutoff"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-march=x86-64-v3", "-o", str(exe),
                    str(ROOT / "tools" / "check_cutoff.cpp")], check=True, capture_output=True)
    res = subprocess.run([str(exe), "quick"], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.strip().endswith("ok")


def test_bench_reference_arm_never_loads_the_product_library():
    """VERDICT r1 #10: `bench.py --impl reference` is the CPU port alone; libs2cuda.so must not be mapped."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, LD_DEBUG="files")
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, env=env, timeout=600)
    assert res.returncode == 0
    assert "libs2cuda" not in res.stderr and "libs2cuda" not in res.stdout
    assert '"impl": "reference"' in res.stdout


def test_patch_example_is_the_default_patch():
    p = s2patch.parse(EXAMPLE_SYNTH2)
    assert p.name == "mySynth" and p.filter_kind == s2.FILTER_ONE_POLE and p.events.size == 0
    assert p.voice.tobytes() == s2.default_voice(1)[0].tobytes()
    assert s2patch.default_patch().voice.tobytes() == p.voice.tobytes()


def test_patch_fields_follow_static_config_layer():
    p = s2patch.parse("""
        // every field of static_config::Layer
        synth lead {
            osc { kind triangle; gain 0.75 }
            noise 0.125                       # Unipolar<1>
            lpf { freq 1200; kind biquad; damping 0.5 }
            amp_env { attack 5; decay 50; sustain 0.625; release 300 }
            mod_env { attack 1 decay 100 sustain 0.25 release 10 }
            modulations { mod_env_to_osc_freq -0.5; mod_env_to_lpf_freq 1.5 }
        }
        score {
            on 0 69
            on 0.5s 72 0.5
            off 1s 69;  off 1500ms 72
        }
    """, sample_rate=48000)
    v = p.voice
    assert p.name == "lead" and p.filter_kind == s2.FILTER_BIQUAD_LP
    assert v["osc_kind"] == s2.OSC_TRIANGLE and v["osc_gain"] == 0.75 and v["noise_amt"] == 0.125
    assert v["lpf_freq_hz"] == 1200.0 and v["damping"] == 0.5
    assert [v[k] for k in ("amp_attack_ms", "amp_decay_ms", "amp_sustain", "amp_release_ms")] == [5.0, 50.0, 0.625, 300.0]
    assert [v[k] for k in ("mod_attack_ms", "mod_decay_ms", "mod_sustain", "mod_release_ms")] == [1.0, 100.0, 0.25, 10.0]
    assert v["mod_env_to_osc_freq"] == -0.5 and v["mod_env_to_lpf_freq"] == 1.5
    assert list(p.events["frame"]) == [0, 24000, 48000, 72000]
    assert list(p.events["note"]) == [69, 72, 69, 72] and list(p.events["on"]) == [1, 1, 0, 0]
    assert list(p.events["velocity"][:2]) == [1.0, 0.5]
    # the same score at another rate
    assert list(s2patch.parse("synth a { } score { on 10ms 60; off 1s 60 }", 44100).events["frame"]) == [441, 44100]


@pytest.mark.parametrize("text,needle", [
    ("synth x { osc { kind pulse } }", "unknown oscillator 'pulse'"),
    ("synth x { noise 2 }", "outside [0, 1]"),                          # units.rs:55-65 range checks
    ("synth x { modulations { mod_env_to_lpf_freq 11 } }", "outside [-10, 10]"),
    ("synth x {\n  lpf { freq 100 }\n  reverb 1\n}", "line 3: unknown field reverb"),
    ("synth x {", "expected '}'"),
    ("score { on 0 69 }", "no synth block"),
    ("synth x { } synth y { }", "more than one synth block"),
    ("synth x { } score { on 10 69; off 5 69 }", "time order"),
    ("synth x { } score { on 0 128 }", "MIDI note"),
    ("synth x { } score { on 1.5 60 }", "whole number of frames"),
    ("synth x { lpf { freq 10kHz } }", "unknown unit"),
    ("synth x { amp_env { sustain 1.5 } }", "amp_env.sustain"),
])
def test_patch_errors_name_the_line_and_field(text, needle):
    with pytest.raises(s2.S2Error) as e:
        s2patch.parse(text)
    assert needle in str(e.value) and "patch line" in str(e.value)


def test_patch_text_round_trip():
    src = """synth lead { osc { kind sine; gain 0.3 } noise 0.0625
        lpf { freq 1234.5; kind biquad_bp; damping 3.25 }
        amp_env { attack 0.1; decay 33.3; sustain 0.7; release 250 }
        mod_env { attack 2; decay 60; sustain 0.1; release 9 }
        modulations { mod_env_to_osc_freq 0.25; mod_env_to_lpf_freq -2.5 } }
        score { on 0 60 0.8; on 480 64; off 4800 60; off 9600 64 }"""
    p = s2patch.parse(src)
    q = s2patch.parse(s2patch.dumps(p))
    assert q.record.tobytes() == p.record.tobytes()
    assert q.events.tobytes() == p.events.tobytes()
    d = s2patch.parse(s2patch.dumps(s2patch.default_patch()))
    assert d.voice.tobytes() == s2.default_voice(1)[0].tobytes() and d.name == "patch"


def test_patch_struct_layouts():
    assert s2.PATCH.itemsize == 144 and s2.PATCH.fields["filter_kind"][1] == 80 and s2.PATCH.fields["name"][1] == 84
    assert s2.NOTE_EVENT.itemsize == 16 and s2.NOTE_EVENT.fields["velocity"][1] == 12
    assert re.search(r"char name\[60\];", HEADER) and re.search(r"\} s2_note_event;\s+/\* 16 bytes \*/", HEADER)


def test_wav_writer_roundtrip(tmp_path):
    from synth2_b200.render import write_wav_f32
    x = np.linspace(-1, 1, 1000, dtype=np.float32)
    path = tmp_path / "x.wav"
    write_wav_f32(path, x, 48000)
    raw = path.read_bytes()
    assert raw[:4] == b"RIFF" and raw[8:12] == b"WAVE" and int.from_bytes(raw[4:8], "little") == len(raw) - 8
    i = raw.index(b"data")
    assert int.from_bytes(raw[i + 4:i + 8], "little") == 4000
    assert np.frombuffer(raw[i + 8:], dtype="<f4").tobytes() == x.tobytes()


# ---- the C ABI from compiled code (examples/render_patch.cpp) ---------------------------------

def build_example(tmp_path):
    exe = tmp_path / "render_patch"
    cmd = ["g++", "-std=c++17", "-O1", f"-I{ROOT / 'include'}", str(ROOT / "examples" / "render_patch.cpp"),
           f"-L{ROOT / 'synth2_b200'}", "-ls2cuda", f"-Wl,-rpath,{ROOT / 'synth2_b200'}", "-o", str(exe)]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr
    return exe


def test_compiled_example_links_and_fails_loudly_without_a_gpu(tmp_path):
    exe = build_example(tmp_path)
    (tmp_path / "p.synth2").write_text(EXAMPLE_SYNTH2)
    res = subprocess.run([str(exe), str(tmp_path / "p.synth2"), "0.01", "48000", str(tmp_path / "o.f32")],
                         capture_output=True, text=True)
    import torch
    if torch.cuda.is_available():
        assert res.returncode == 0, res.stderr
    else:
        assert res.returncode == 1 and "no CUDA device" in res.stderr       # no CPU path, said plainly
    bad = subprocess.run([str(exe), str(tmp_path / "missing.synth2"), "1", "48000", str(tmp_path / "o.f32")],
                         capture_output=True, text=True)
    assert bad.returncode == 2
