"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol that
include/stratum_b200.h declares, the struct mirrors match, the pure-host entry points
(config_default, compute_confidence, warning strings, key names) agree with the oracle, and compute
entry points fail loudly without a CUDA device (no CPU fallback)."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

import oracle_lib as O
import stratum_dsp_b200 as S

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()


def declared_symbols():
    return sorted(set(re.findall(r"\b(stratum_b200_[a-z0-9_]+)\s*\(", HEADER)))


def test_header_symbols_are_exported():
    L = S.lib()
    syms = declared_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/stratum_b200.h but not exported"


def test_struct_sizes_match():
    L = S.lib()
    assert L.stratum_b200_sizeof(0) == C.sizeof(S.StratumConfig)
    assert L.stratum_b200_sizeof(1) == C.sizeof(S.StratumResult)
    assert L.stratum_b200_sizeof(2) == C.sizeof(S.StratumConfidence)
    # every config field of the header is mirrored, in order
    body = HEADER[HEADER.index("typedef struct StratumConfig {") + len("typedef struct StratumConfig {"):HEADER.index("} StratumConfig;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        m = re.match(r"(uint32_t|int32_t|float)\s+(.*)$", decl, flags=re.S)
        if m:
            names += [re.sub(r"\[.*\]", "", n).strip() for n in m.group(2).split(",")]
    assert names == [n for n, _ in S.StratumConfig._fields_]


def test_config_default_matches_reference_defaults():
    # src/config.rs:594-744 through the oracle's Config (same source of truth, separately typed in)
    L = O.lib()
    oc = L.so_config_new()
    c = S.AnalysisConfig()
    checked = 0
    for name, _ in S.StratumConfig._fields_:
        v = L.so_config_get(oc, name.encode())
        if np.isnan(v):
            continue
        assert float(getattr(c, name)) == pytest.approx(v, rel=1e-7), name
        checked += 1
    L.so_config_free(oc)
    assert checked >= 70
    assert c.onset_consensus_weights == [0.25] * 4 and c.abi_version == S.ABI_VERSION
    assert c.enable_hpss_onsets == 0 and c.enable_bpm_fusion == 0 and c.enable_key_mode_heuristic == 0


def test_config_rejects_unknown_fields():
    with pytest.raises(AttributeError):
        S.AnalysisConfig(no_such_field=1)


def test_key_names():
    assert S.Key(False, 0).name() == "C" and S.Key(False, 6).name() == "F#" and S.Key(True, 9).name() == "Am"
    assert S.Key(False, 0).numerical() == "1A" and S.Key(False, 7).numerical() == "2A"
    assert S.Key(True, 9).numerical() == "1B" and S.Key(True, 4).numerical() == "2B"
    L = O.lib()
    for minor in (0, 1):
        for i in range(12):
            for num in (0, 1):
                b = C.create_string_buffer(16)
                L.so_key_name(minor, i, num, b, 16)
                k = S.Key(bool(minor), i)
                assert (k.numerical() if num else k.name()) == b.value.decode()


@pytest.mark.parametrize("seed", range(40))
def test_compute_confidence_matches_oracle(seed):
    rng = np.random.default_rng(seed)
    bpm = float(rng.choice([0.0, 90.0, 128.0]))
    vals = [float(rng.uniform(-0.2, 1.3)) for _ in range(4)]
    warn = int(rng.integers(0, 16))
    flags = int(rng.integers(0, 16))
    r = S.StratumResult()
    r.bpm, r.bpm_confidence, r.key_confidence, r.key_clarity, r.grid_stability = bpm, *vals
    r.warnings, r.flags = warn, flags
    out = S.StratumConfidence()
    S.lib().stratum_b200_compute_confidence(C.byref(r), C.byref(out))
    exp = (C.c_float * 4)()
    fl = C.c_uint32()
    O.lib().so_confidence_of(bpm, *vals, warn, flags, exp, C.byref(fl))
    assert [out.bpm_confidence, out.key_confidence, out.grid_stability, out.overall_confidence] == list(exp)
    assert out.flags == fl.value


def test_warning_strings_are_the_reference_strings():
    r = S.StratumResult()
    r.warnings = 15
    r.grid_stability, r.key_confidence, r.key_clarity = 0.123, 0.256, 0.1
    buf = C.create_string_buffer(1024)
    S.lib().stratum_b200_warning_strings(C.byref(r), buf, 1024)
    lines = buf.value.decode().strip().split("\n")
    assert lines == [  # src/lib.rs:1567-1589
        "BPM detection failed: insufficient onsets or estimation error",
        "Low beat grid stability: 0.12 (may indicate tempo variation)",
        "Low key detection confidence: 0.26 (may indicate ambiguous or atonal music)",
        "Low key clarity: 0.10 (track may be atonal or have weak tonality)",
    ]


def test_metadata_literals_are_the_reference_literals():
    # AnalysisMetadata fields the wrappers synthesise (the C result carries the numbers): quoted from the reference
    assert S.ALGORITHM_VERSION == "0.1.0-alpha"  # src/lib.rs:1603
    assert list(S.METHODS_USED) == ["energy_flux", "chroma_extraction", "key_detection"]  # src/lib.rs:1604-1608
    rs = (ROOT / "rust" / "stratum-dsp-b200" / "src" / "lib.rs").read_text()
    assert 'vec!["energy_flux".to_string(), "chroma_extraction".to_string(), "key_detection".to_string()]' in rs
    assert 'algorithm_version: "0.1.0-alpha".to_string()' in rs
    # flag order of AnalysisFlag (src/analysis/result.rs) as the wrappers emit it
    assert [n for _, n in sorted(S._FLAG_NAMES.items())] == ["MultimodalBpm", "WeakTonality", "TempoVariation", "OnsetDetectionAmbiguous"]


def test_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    with pytest.raises(S.AnalysisError) as e:
        S.analyze_audio(np.ones(4096, np.float32), 44100)
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message
    with pytest.raises(S.AnalysisError):
        S.stft(np.ones(4096, np.float32), 2048, 512)


def test_config_validation_happens_before_any_device_work():
    # rejected switches give NotImplemented even on a box without a GPU
    for kw in ({"enable_hpss_onsets": 1, "hpss_margin": 11}, {"key_multi_scale_n_lengths": 9}, {"key_hpcp_peaks_per_frame": 64}, {"frame_size": 1024}, {"hop_size": 16}, {"hop_size": 40000}, {"key_stft_frame_size": 3000}, {"key_stft_frame_size": 16384}, {"tempogram_multi_res_top_k": 64},
               {"key_hpss_time_margin": 11, "enable_key_hpss_harmonic": 1}):
        with pytest.raises(S.AnalysisError) as e:
            S.analyze_batch([np.ones(4096, np.float32)], 44100, S.AnalysisConfig(**kw))
        assert e.value.kind == "NotImplemented", kw
    with pytest.raises(S.AnalysisError) as e:
        S.analyze_batch([np.ones(4096, np.float32)], 44100, S.AnalysisConfig(min_bpm=200.0, max_bpm=100.0))
    assert e.value.kind == "InvalidInput"
    with pytest.raises(S.AnalysisError) as e:
        S.analyze_batch([np.ones(4096, np.float32)], 44100, S.AnalysisConfig(hop_size=0))
    assert e.value.kind == "InvalidInput"


def test_product_does_not_touch_the_oracle():
    # the shipped package never imports, links or executes anything under oracle/
    for p in (ROOT / "stratum_dsp_b200").rglob("*"):
        if p.suffix in {".py", ".cu", ".cuh", ".h"} or p.name == "Makefile":
            txt = p.read_text()
            assert "oracle_lib" not in txt and "libstratum_oracle" not in txt and "so_common.hpp" not in txt, p
    import subprocess
    out = subprocess.run(["ldd", str(S.LIB_PATH)], capture_output=True, text=True).stdout
    assert "oracle" not in out


def test_rust_binding_is_generated_from_the_header():
    # rust/stratum-dsp-b200/src/sys.rs mirrors include/stratum_b200.h field for field (the crate ships as source: no Rust toolchain here)
    import subprocess
    import sys
    assert subprocess.run([sys.executable, str(ROOT / "tools" / "gen_rust_sys.py"), "--check"]).returncode == 0, "run tools/gen_rust_sys.py"
    rs = (ROOT / "rust" / "stratum-dsp-b200" / "src" / "sys.rs").read_text()
    names = [n for n, _ in S.StratumConfig._fields_]
    got = re.findall(r"pub (\w+):", rs[rs.index("pub struct StratumConfig {"):rs.index("pub struct StratumTempoCandidate {")])
    assert got == names
    wrapper = (ROOT / "rust" / "stratum-dsp-b200" / "src" / "lib.rs").read_text()
    for sym in re.findall(r"(stratum_b200_\w+)\(", wrapper):
        assert sym in HEADER and f"pub fn {sym}(" in rs, sym


def _plan(lens, srs=None, budget_gb=100.0, cfg=None):
    L = S.lib()
    L.stratum_b200_debug_plan_waves.restype = C.c_uint32
    n = len(lens)
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum(np.asarray(lens, np.uint64))
    sr = np.full(n, 44100, np.uint32) if srs is None else np.asarray(srs, np.uint32)
    out = np.zeros(n, np.uint32)
    nw = L.stratum_b200_debug_plan_waves(off.ctypes.data_as(C.POINTER(C.c_uint64)), sr.ctypes.data_as(C.POINTER(C.c_uint32)), n,
                                         C.byref(cfg._c) if cfg else None, C.c_double(budget_gb), out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return nw, out


def test_wave_planner_balances_and_respects_the_budget():
    T3 = 7_938_000  # 3 minutes at 44.1 kHz
    nw, w = _plan([T3] * 1024)                      # wave cap = 208 three-minute tracks: five even waves
    assert nw == 5 and sorted(np.bincount(w).tolist()) == [204, 205, 205, 205, 205]
    nw, w = _plan([T3] * 215)                       # a little over one full wave: two balanced waves, not 208 + 7
    assert nw == 2 and sorted(np.bincount(w).tolist()) == [107, 108]
    nw, w = _plan([T3] * 64)
    assert nw == 1
    nw, w = _plan([T3 // 6] * 3000)                 # short tracks: the cap is in samples, not in tracks
    assert nw == 3 and np.bincount(w).min() >= 900
    nw, w = _plan([T3] * 200, budget_gb=10.0)       # a 10 GB arena holds ~25 three-minute tracks with their escalation room
    assert nw >= 8 and np.bincount(w).max() <= 32 and np.all(np.diff(w) >= 0)
    rng = np.random.RandomState(3)
    lens = (np.exp(rng.uniform(np.log(30), np.log(600), 256)) * 44100).astype(np.uint64)   # C5: ragged 30 s - 10 min
    nw, w = _plan(lens, srs=[44100, 48000] * 128)
    assert np.all(np.diff(w) >= 0) and w[0] == 0 and w[-1] == nw - 1                       # contiguous, in order, every track placed
    per = [int(lens[w == k].sum()) for k in range(nw)]
    assert max(per) <= 1.5 * 208 * T3 and (nw == 1 or min(per) >= 0.3 * max(per))          # no tiny tail wave
    nw, w = _plan([200 * T3])                       # one 10-hour track: still planned (the budget is raised for a single track)
    assert nw == 1
    # hop_size other than 512 gives the base path a slot of its own (more frames at a smaller hop): the same budget holds fewer tracks
    nw512, _ = _plan([T3] * 200, budget_gb=20.0)
    nw128, w = _plan([T3] * 200, budget_gb=20.0, cfg=S.AnalysisConfig(hop_size=128))
    nw2048, _ = _plan([T3] * 200, budget_gb=20.0, cfg=S.AnalysisConfig(hop_size=2048))
    assert nw128 > nw2048 >= nw512 and np.all(np.diff(w) >= 0)


def test_mel_fold_schedule_partitions_every_band():
    # par_feat_kernel folds the mel triangles as <= 64 chunks of the bands' entry lists, two per lane, then adds each band's partial sums
    # in order (period/novelty.rs:172-189 accumulates per band in ascending-bin order; the curve is a tolerance-level quantity)
    L = S.lib()
    L.stratum_b200_debug_mel_schedule.restype = None
    rng = np.random.RandomState(11)
    cases = [np.array([0] + list(np.cumsum(rng.randint(1, 120, nm))), np.int32) for nm in (4, 17, 40, 40)]
    cases.append(np.array([0] + list(np.cumsum([2, 2, 3, 3] + list(range(3, 39)))), np.int32))   # the shape of a real filterbank: widening triangles
    cases.append(np.zeros(1, np.int32))                                                            # mel novelty off
    for off in cases:
        nm = len(off) - 1
        ck = np.full(256, -7, np.int32)
        L.stratum_b200_debug_mel_schedule(off.ctypes.data_as(C.POINTER(C.c_int32)), nm, ck.ctypes.data_as(C.POINTER(C.c_int32)))
        a, e, pos, band0 = ck[:64], ck[64:128], ck[128:192], ck[192:233]
        live = [i for i in range(64) if e[i] > a[i]]
        assert sorted(pos.tolist()) == list(range(64)) or len(set(pos[live].tolist())) == len(live)   # one partial-sum slot per live chunk
        lens = (e - a)[live]
        assert np.all(np.diff(lens) <= 0)                                                          # longest first: the first 32 are round one
        n_chunks = len(live)
        assert n_chunks <= 64 and band0[nm] == n_chunks and np.all(band0[nm:] == n_chunks)
        by_pos = {int(pos[i]): (int(a[i]), int(e[i])) for i in live}
        for m in range(nm):                                                                        # a band's chunks, in position order, tile its entry range
            cur = int(off[m])
            for p in range(int(band0[m]), int(band0[m + 1])):
                assert by_pos[p][0] == cur
                cur = by_pos[p][1]
            assert cur == int(off[m + 1])
        if n_chunks:
            total = int(off[-1])
            assert lens.max() <= -(-total // 64) * 2 + max(1, int(np.diff(off).min()))              # balanced: no chunk much longer than the mean
        idle = [i for i in range(64) if i not in live]
        assert all(int(pos[i]) >= n_chunks for i in idle)                                          # idle slots write where no band reads


def test_division_by_25_is_exact_for_every_float(tmp_path):
    # tools/check_div_by_const.c: RN(a * RN(1/25)) corrected once (csrc/common.cuh div_by_25_rn) equals a / 25.0f for every finite
    # float with |a| >= 1e-30 — exhaustive over all 2^32 bit patterns (about 20 s on 8 threads)
    import subprocess
    exe = tmp_path / "div25"
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-mfma", "-o", str(exe), str(ROOT / "tools" / "check_div_by_const.c"), "-lm", "-lpthread"], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout
    assert "mismatches with |a| >= 1e-30: 0" in out, out


@pytest.mark.parametrize("fmt,ext,ch", [("s16", False, 1), ("s24", False, 2), ("s32", True, 6), ("u8", False, 1), ("f32", True, 2), ("f64", False, 3)])
def test_wav_container_reader(tmp_path, fmt, ext, ch):
    # host half of the decoder-side entry: the RIFF/WAVE container is parsed without touching the samples (stratum_dsp_b200.read_wav)
    import wavgen
    rng = np.random.default_rng(7)
    x = (rng.standard_normal((1234, ch)) * 0.2).squeeze()
    p = tmp_path / "t.wav"
    p.write_bytes(wavgen.wav_bytes(x, 48000, fmt, extensible=ext, extra_chunk=True))
    t = S.read_wav(p)
    want = {"u8": S.PCM_U8, "s16": S.PCM_S16, "s24": S.PCM_S24, "s32": S.PCM_S32, "f32": S.PCM_F32, "f64": S.PCM_F64}[fmt]
    assert (t.fmt, t.channels, t.sample_rate, t.frames) == (want, ch, 48000, 1234)
    assert t.data.tobytes() == wavgen.encode(x, fmt)


def test_wav_container_reader_rejects_other_formats(tmp_path):
    import struct
    p = tmp_path / "bad.wav"
    p.write_bytes(b"RIFF" + struct.pack("<I", 36) + b"WAVE" + b"fmt " + struct.pack("<IHHIIHH", 16, 0x55, 2, 44100, 0, 0, 0) + b"data" + struct.pack("<I", 0))
    with pytest.raises(ValueError, match="Unsupported sample format"):
        S.read_wav(p)
    p.write_bytes(b"OggS....")
    with pytest.raises(ValueError):
        S.read_wav(p)
