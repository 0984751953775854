"""The reference's CLI surface on the B200 path (SURVEY §8f n3): flag -> AnalysisConfig mapping of examples/analyze_file.py
against examples/analyze_file.rs:254-690, and the --json document against analyze_file.rs:722-773.  CPU only: building a
configuration and formatting a result need no device."""
import importlib.util
import sys
import wave
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent


def _load(name):
    spec = importlib.util.spec_from_file_location(name, ROOT / "examples" / f"{name}.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


AF = _load("analyze_file")


def test_every_flag_of_the_reference_usage_line_is_known():
    # the usage string of examples/analyze_file.rs:186 lists the flags.  tests/golden/reference_cli_flags.json holds the 119 of them as
    # the mirror's tables recorded them when they were checked against that file ("source" says how): no flag of that set may be dropped
    import json

    known = set(AF.BOOL_FLAGS) | set(AF.VALUE_FLAGS) | AF.IGNORED | AF.IGNORED_WITH_VALUE
    assert set(AF.ORDER) == set(AF.BOOL_FLAGS) | set(AF.VALUE_FLAGS) and len(AF.ORDER) == len(set(AF.ORDER))
    flags = set(json.loads((ROOT / "tests" / "golden" / "reference_cli_flags.json").read_text())["flags"])
    assert len(flags) == 119 and flags <= known, sorted(flags - known)
    assert len(known) >= 115


def test_flags_map_to_the_reference_fields():
    c = AF.build_config([])
    d = __import__("stratum_dsp_b200").AnalysisConfig()
    assert all(getattr(c, n) == getattr(d, n) for n in ("enable_key_hpcp", "key_stft_frame_size", "tempogram_band_seed_only", "enable_normalization"))
    c = AF.build_config(["--no-preprocess", "--bpm-candidates-top", "7", "--band-score-fusion", "--key-hpss-frame-step", "0", "--key-stft-hop-size", "256",
                         "--key-multi-scale-lengths", "100, 300,900", "--key-multi-scale-weights", "0.5,1,2", "--key-template-temperley",
                         "--key-mode-third-margin", "0.25", "--multi-res-w256", "0.4", "--key-hpcp-whitening-smooth-bins", "2", "--legacy-mul-soft", "0.5"])
    assert (c.enable_normalization, c.enable_silence_trimming) == (0, 0)
    assert (c.emit_tempogram_candidates, c.tempogram_candidates_top_n) == (1, 7)
    assert c.tempogram_band_seed_only == 0
    assert (c.enable_key_hpss_harmonic, c.key_hpss_frame_step) == (1, 1)          # n.max(1)
    assert (c.enable_key_stft_override, c.key_stft_hop_size) == (1, 256)
    assert (c.enable_key_multi_scale, c.key_multi_scale_lengths, c.key_multi_scale_weights) == (1, [100, 300, 900], [0.5, 1.0, 2.0])
    assert c.key_template_set == 1
    assert c.enable_key_mode_heuristic == 1 and c.key_mode_third_ratio_margin == pytest.approx(0.25)
    assert c.enable_tempogram_multi_resolution == 1 and c.tempogram_multi_res_w256 == pytest.approx(0.4)
    assert (c.enable_key_hpcp_whitening, c.key_hpcp_whitening_smooth_bins) == (1, 3)  # n.max(3)
    assert c.legacy_bpm_conf_mul_soft == pytest.approx(0.5)
    # later blocks of the reference win: --no-key-hpss after --key-hpss, --key-ensemble after --no-key-ensemble
    c = AF.build_config(["--no-key-hpss", "--key-hpss", "--no-key-ensemble", "--key-ensemble", "--no-key-stft-override", "--key-stft-frame-size", "100"])
    assert c.enable_key_hpss_harmonic == 0 and c.enable_key_ensemble == 1
    assert (c.enable_key_stft_override, c.key_stft_frame_size) == (1, 256)         # explicit size re-enables the override, n.max(256)
    # values that do not parse leave the default (parse().ok())
    c = AF.build_config(["--key-segment-len-frames", "-5", "--mel-weight", "abc"])
    assert c.key_segment_len_frames == 1024 and c.tempogram_mel_weight == pytest.approx(0.15)


def test_json_document_matches_the_reference_format():
    key = SimpleNamespace(name=lambda: "F#m")
    meta = SimpleNamespace(tempogram_multi_res_triggered=True, tempogram_multi_res_used=False, tempogram_percussive_triggered=None,
                           tempogram_percussive_used=None, tempogram_candidates=[(128.0, 0.98765, 1.0, 0.5, True), (64.0, 0.5, 0.25, 0.125, False)],
                           processing_time_ms=1.005)
    r = SimpleNamespace(bpm=np.float32(127.996), key=key, key_clarity=0.61, grid_stability=0.9949, metadata=meta)
    c = SimpleNamespace(bpm_confidence=0.499, key_confidence=0.0)
    assert AF.render_json(r, c) == "\n".join([
        "{", '  "bpm": 128.00,', '  "bpm_confidence": 0.50,', '  "key": "F#m",', '  "key_confidence": 0.00,', '  "key_clarity": 0.61,',
        '  "grid_stability": 0.99,', '  "tempogram_multi_res_triggered": true,', '  "tempogram_multi_res_used": false,', '  "bpm_candidates": [',
        '    { "bpm": 128.00, "score": 0.9877, "fft_norm": 1.0000, "autocorr_norm": 0.5000, "selected": true },',
        '    { "bpm": 64.00, "score": 0.5000, "fft_norm": 0.2500, "autocorr_norm": 0.1250, "selected": false }', "  ],",
        '  "processing_time_ms": 1.00', "}"])


def test_wav_decode_follows_the_reference_arithmetic(tmp_path):
    # S16 stereo: per-channel s/32768, left-to-right f32 sum, / channels (analyze_file.rs:97-110)
    pcm = np.array([[1000, -2000], [32767, 32767], [-32768, 0]], dtype="<i2")
    p = tmp_path / "t.wav"
    with wave.open(str(p), "wb") as w:
        w.setnchannels(2)
        w.setsampwidth(2)
        w.setframerate(48000)
        w.writeframes(pcm.tobytes())
    x, sr = AF.decode_wav(str(p))
    exp = (pcm[:, 0].astype(np.float32) / np.float32(32768) + pcm[:, 1].astype(np.float32) / np.float32(32768)) / np.float32(2)
    assert sr == 48000 and x.dtype == np.float32 and np.array_equal(x, exp)


@pytest.mark.gpu
def test_analyze_file_cli_end_to_end(tmp_path):
    # the script a validation harness would call instead of the Rust binary: WAV in, the reference's JSON document out
    import json
    import subprocess

    import stratum_dsp_b200 as S
    import synth

    x = synth.render(synth.c2_params(21, 12 * 44100, 44100))
    pcm = np.clip(np.round(x.astype(np.float64) * 32768.0), -32768, 32767).astype("<i2")
    p = tmp_path / "track.wav"
    with wave.open(str(p), "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(44100)
        w.writeframes(pcm.tobytes())
    flags = ["--json", "--bpm-candidates-top", "5", "--key-template-temperley", "--no-trim"]
    out = subprocess.run([sys.executable, str(ROOT / "examples" / "analyze_file.py"), str(p)] + flags, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    doc = json.loads(out.stdout)
    r = S.analyze_audio(pcm.astype(np.float32) / np.float32(32768.0), 44100, AF.build_config(flags))
    c = S.compute_confidence(r)
    assert doc["bpm"] == float(f"{r.bpm:.2f}") and doc["key"] == r.key.name()
    assert doc["bpm_confidence"] == float(f"{c.bpm_confidence:.2f}") and doc["grid_stability"] == float(f"{r.grid_stability:.2f}")
    assert len(doc["bpm_candidates"]) == len(r.metadata.tempogram_candidates) >= 1
    assert [cd["selected"] for cd in doc["bpm_candidates"]] == [bool(t[4]) for t in r.metadata.tempogram_candidates]
    assert list(doc)[:6] == ["bpm", "bpm_confidence", "key", "key_confidence", "key_clarity", "grid_stability"] and list(doc)[-1] == "processing_time_ms"


def _build_cpp_example():
    import subprocess

    subprocess.run(["make", "-s", "-C", str(ROOT / "stratum_dsp_b200"), "example"], check=True)
    return ROOT / "stratum_dsp_b200" / "_build" / "analyze_batch"


def _write_wav(path, x, sr=44100, channels=1):
    pcm = np.clip(np.round(np.asarray(x, np.float64) * 32768.0), -32768, 32767).astype("<i2")
    with wave.open(str(path), "wb") as w:
        w.setnchannels(channels)
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(pcm.tobytes())
    return pcm


def test_cpp_example_links_against_the_c_abi_and_fails_loudly_without_a_device(tmp_path):
    # compiled host code over include/stratum_b200.h alone (what a Rust / Go / Java binding would link): builds, prints usage,
    # and on a box without a GPU reports the library's error instead of computing anything on the CPU
    import subprocess

    import stratum_dsp_b200 as S

    exe = _build_cpp_example()
    assert subprocess.run([str(exe), "--help"], capture_output=True, text=True).returncode == 0
    if S.device_count() == 0:
        _write_wav(tmp_path / "a.wav", 0.3 * np.sin(2 * np.pi * 440 * np.arange(44100) / 44100))
        out = subprocess.run([str(exe), "--json", str(tmp_path / "a.wav")], capture_output=True, text=True)
        assert out.returncode == 1 and "no CPU fallback" in out.stderr and out.stdout == ""


@pytest.mark.gpu
def test_cpp_example_matches_the_python_mirror(tmp_path):
    import json
    import subprocess

    import stratum_dsp_b200 as S
    import synth

    exe = _build_cpp_example()
    xs = [synth.render(synth.c2_params(31, 10 * 44100, 44100)), synth.render(synth.c2_params(32, 8 * 44100, 44100))]
    pcms = [_write_wav(tmp_path / f"t{i}.wav", x) for i, x in enumerate(xs)]
    out = subprocess.run([str(exe), "--json"] + [str(tmp_path / f"t{i}.wav") for i in range(2)] + [str(tmp_path / "missing.wav")], capture_output=True, text=True)
    lines = [json.loads(l) for l in out.stdout.splitlines()]
    assert len(lines) == 3 and out.returncode == 1                      # one file could not be read: reported per item, the batch went on
    assert lines[2]["file"].endswith("missing.wav") and lines[2]["error"].startswith("decode failed:")
    for doc, pcm in zip(lines, pcms):
        r = S.analyze_audio(pcm.astype(np.float32) / np.float32(32768.0), 44100)
        c = S.compute_confidence(r)
        assert doc["bpm"] == float(f"{r.bpm:.2f}") and doc["key"] == r.key.name() and doc["bpm_confidence"] == float(f"{c.bpm_confidence:.4f}")
        assert list(doc) == ["file", "bpm", "bpm_confidence", "key", "key_confidence", "processing_time_ms", "tempogram_multi_res_triggered",
                             "tempogram_multi_res_used", "tempogram_percussive_triggered", "tempogram_percussive_used"]
