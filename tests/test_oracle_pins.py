"""Pins the CPU oracle to every known answer the reference's own tests hold for this path
(SURVEY.md §8c).  The Rust reference cannot be built here, so these are the anchors."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import synth


# ---- tests/integration_tests.rs:46-275 on re-created fixtures (scripts/generate_fixtures.py) ----------
def test_fixture_120bpm():
    r = O.analyze(synth.fixture_kick(120.0, 8.0), 44100)
    assert r.status == 0
    if r.bpm > 0:
        assert abs(r.bpm - 120.0) <= 2.0  # integration_tests.rs:62-67


def test_fixture_128bpm():
    r = O.analyze(synth.fixture_kick(128.0, 7.5), 44100)
    assert r.status == 0
    if r.bpm > 0:
        assert abs(r.bpm - 128.0) <= 2.0  # :141-146


def test_fixture_cmajor_scale():
    r = O.analyze(synth.fixture_cmajor_scale(), 44100)
    assert r.status == 0
    assert (r.key == 0) or r.key_confidence < 0.3  # :209-213


def test_fixture_mixed_silence_trim():
    r = O.analyze(synth.fixture_mixed_silence(), 44100)
    assert r.status == 0
    assert 4.0 <= r.duration_seconds <= 6.0  # :246-250


def test_all_silence_is_an_error():
    r = O.analyze(np.zeros(44100, np.float32), 44100)
    assert r.status == 3 and "silent" in r.error  # :264-274


def test_empty_and_bad_rate():
    assert O.analyze(np.zeros(0, np.float32), 44100).status == 1  # lib.rs:100-104
    assert O.analyze(np.ones(10, np.float32), 0).status == 1  # lib.rs:106-110


def test_criterion_bench_shape_returns():
    # benches/audio_analysis_bench.rs:25-29, 410-423: 30 s 440 Hz sine x 0.5 must analyse without error
    sr = 44100
    x = (0.5 * np.sin(2 * np.pi * 440.0 * np.arange(30 * sr) / sr)).astype(np.float32)
    assert O.analyze(x, sr).status == 0


# ---- unit-test known answers -----------------------------------------------------------------------------
def test_consensus_known_answer():
    # onset/consensus.rs:293-308: four methods agreeing on 1000 -> one cluster at 1000 voted by 4
    L = O.lib()
    a = np.array([1000], np.int64)
    centre, conf, voted = np.zeros(8, np.int64), np.zeros(8, np.float32), np.zeros(8, np.uint32)
    w = np.full(4, 0.25, np.float32)
    n = L.so_vote_onsets(O.i64ptr(a), 1, O.i64ptr(a), 1, O.i64ptr(a), 1, O.i64ptr(a), 1, O.f32ptr(w), 50, 44100, O.i64ptr(centre), O.f32ptr(conf),
                         voted.ctypes.data_as(C.POINTER(C.c_uint32)), 8)
    assert n == 1 and centre[0] == 1000 and voted[0] == 4 and abs(conf[0] - 1.0) < 1e-6


def test_key_templates_and_detection():
    # key/detector.rs:1014-1048: C-E-G chroma -> Key::Major(0); :1069-1075 dot = 32 is plain arithmetic
    L = O.lib()
    chroma = np.zeros((10, 12), np.float32)
    chroma[:, [0, 4, 7]] = [1.0, 0.8, 0.9]
    key, conf, clar = C.c_int(), C.c_float(), C.c_float()
    st = L.so_detect_key(O.f32ptr(chroma), 10, None, C.byref(key), C.byref(conf), C.byref(clar), None, None)
    assert st == 0 and key.value == 0
    maj, mnr = np.zeros(144, np.float32), np.zeros(144, np.float32)
    L.so_key_templates(O.f32ptr(maj), O.f32ptr(mnr))
    maj = maj.reshape(12, 12)
    assert np.allclose(np.linalg.norm(maj, axis=1), 1.0, atol=1e-6)
    assert np.allclose(maj[3], np.roll(maj[0], 3))  # templates.rs:88-101 rotation


def test_key_clarity_known_answers():
    # key/key_clarity.rs:100-148: clear winner -> high clarity; flat scores -> 0; < 2 scores -> 0
    L = O.lib()
    s = np.array([1.0] + [0.1] * 23, np.float32)
    assert L.so_key_clarity(O.f32ptr(s), 24) > 0.9
    flat = np.full(24, 0.5, np.float32)
    assert L.so_key_clarity(O.f32ptr(flat), 24) == 0.0
    assert L.so_key_clarity(O.f32ptr(s), 1) == 0.0


def test_key_naming_tables():
    # analysis/result.rs:272-369
    L = O.lib()

    def nm(minor, idx, num):
        b = C.create_string_buffer(16)
        L.so_key_name(minor, idx, num, b, 16)
        return b.value.decode()

    assert [nm(0, 0, 0), nm(0, 6, 0), nm(1, 9, 0), nm(1, 1, 0)] == ["C", "F#", "Am", "C#m"]
    assert [nm(0, 0, 1), nm(0, 7, 1), nm(1, 9, 1), nm(1, 4, 1), nm(0, 5, 1), nm(1, 2, 1)] == ["1A", "2A", "1B", "2B", "12A", "12B"]


def test_confidence_known_answers():
    # analysis/confidence.rs:340-422
    L = O.lib()

    def conf(bpm, bc, kc, clar, gs, warn=0, flags=0):
        out = (C.c_float * 4)()
        fl = C.c_uint32()
        L.so_confidence_of(bpm, bc, kc, clar, gs, warn, flags, out, C.byref(fl))
        return list(out), fl.value

    (b, k, g, o), fl = conf(120.0, 0.85, 0.75, 0.7, 0.9)  # high-confidence case
    assert abs(b - 0.85) < 1e-6 and abs(k - 0.75) < 1e-6 and abs(g - 0.9) < 1e-6
    assert abs(o - (0.85 * 0.4 + 0.75 * 0.3 + 0.9 * 0.3)) < 1e-6 and fl == 0
    (b, k, g, o), fl = conf(0.0, 0.0, 0.0, 0.0, 0.0)  # everything failed
    assert (b, k, g, o) == (0.0, 0.0, 0.0, 0.0) and fl == (1 | 2 | 4)
    (b, k, g, o), fl = conf(120.0, 0.8, 0.6, 0.1, 0.8, warn=8)  # low clarity + clarity warning: x0.6 x0.7
    assert abs(k - 0.6 * 0.6 * 0.7) < 1e-6


def test_time_signature_short_list_defaults_to_4_4():
    # beat_tracking/time_signature.rs:246-255: fewer than 8 beats -> 4/4
    L = O.lib()
    on = np.arange(0, 3.0, 0.5, dtype=np.float32)
    stab, nb, nd, bpb = C.c_float(), C.c_int(), C.c_int(), C.c_int()
    st = L.so_beat_grid(120.0, 0.9, O.f32ptr(on), on.size, 44100, C.byref(stab), C.byref(nb), C.byref(nd), C.byref(bpb))
    assert st == 0 and bpb.value == 4 and nb.value == 6


def test_hmm_on_a_clean_grid():
    # beat_tracking/hmm.rs:500-560: onsets exactly on a 120 BPM grid -> every frame kept, frames 0..n-1
    L = O.lib()
    on = (np.arange(16) * 0.5).astype(np.float32)
    fr, tm = np.zeros(64, np.int32), np.zeros(64, np.float32)
    path, plen = np.zeros(64, np.int32), C.c_int()
    n = L.so_hmm(120.0, O.f32ptr(on), 16, fr.ctypes.data_as(C.POINTER(C.c_int32)), O.f32ptr(tm), 64, path.ctypes.data_as(C.POINTER(C.c_int)), 64,
                 C.byref(plen))
    assert n == 16 and list(fr[:16]) == list(range(16)) and plen.value == 16
    assert np.allclose(tm[:16], on, atol=1e-6)


def test_silent_normalisation_is_a_noop():
    # preprocessing/normalization.rs:669-683: silent input -> gain leaves samples untouched (gain 1)
    L = O.lib()
    x = np.zeros(4096, np.float32)
    g, ts, te = C.c_float(), C.c_uint64(), C.c_uint64()
    assert L.so_preprocess(O.f32ptr(x), x.size, 44100, 0, C.byref(g), C.byref(ts), C.byref(te)) == 0
    assert g.value == 1.0 and te.value == 0  # fully silent -> empty trim range


def test_oracle_is_deterministic_and_build_independent():
    p = synth.c2_params(3, 10 * 44100)
    x = synth.render(p)
    a, b = O.analyze(x, 44100), O.analyze(x, 44100, fast=True)
    assert a.bpm == b.bpm and a.key == b.key and a.key_clarity == b.key_clarity and np.array_equal(a.beats, b.beats)


def test_hpss_known_answers():
    # onset/hpss.rs:379-420: constant spectrogram -> harmonic + percussive reconstruct the input; empty input is an error
    L = O.lib()
    spec = np.full((10, 64), 0.5, np.float32)
    h, p = np.zeros_like(spec), np.zeros_like(spec)
    assert L.so_hpss_decompose(O.f32ptr(spec), 10, 64, 5, O.f32ptr(h), O.f32ptr(p)) == 0
    assert np.abs(h + p - spec).max() < 0.1 and np.allclose(h, 0.25) and np.allclose(p, 0.25)
    assert L.so_hpss_decompose(O.f32ptr(spec), 0, 64, 5, O.f32ptr(h), O.f32ptr(p)) == 1
    # a percussive burst (one bright frame) ends up in the percussive part and is picked as an onset at that frame
    spec = np.full((40, 64), 0.01, np.float32)
    spec[20] = 1.0
    h, p = np.zeros_like(spec), np.zeros_like(spec)
    assert L.so_hpss_decompose(O.f32ptr(spec), 40, 64, 10, O.f32ptr(h), O.f32ptr(p)) == 0
    assert p[20].sum() > 10 * h[20].sum()
    on = np.zeros(8, np.int64)
    n = L.so_hpss_onsets(O.f32ptr(p), 40, 64, 0.8, O.i64ptr(on), 8)
    assert n >= 1 and 20 in on[:n]
    # a steady tone (one bright bin) stays harmonic
    spec = np.full((40, 64), 0.01, np.float32)
    spec[:, 30] = 1.0
    assert L.so_hpss_decompose(O.f32ptr(spec), 40, 64, 10, O.f32ptr(h), O.f32ptr(p)) == 0
    assert h[:, 30].sum() > 10 * p[:, 30].sum()


def test_tuning_estimate_recovers_a_known_detune():
    # estimate_tuning_offset_semitones_from_spectrogram (chroma/extractor.rs:66-170) has no unit test in the reference; its
    # intent is checkable: material detuned by +/-30 cents must come out near +/-0.3 semitones, and the clamp of
    # lib.rs:1109-1113 must hold it at key_tuning_max_abs_semitones
    import synth

    for cents in (30.0, -30.0):
        x = synth.render_progression(7, 12, 44100, tonic=0, minor=False, bpm=120, detune_cents=cents)
        o = O.analyze(x, 44100, {"enable_key_tuning_compensation": 1, "key_tuning_max_abs_semitones": 0.5}, dump=True, fast=True)
        t = float(o.farray("key.tuning")[0])
        assert abs(t - cents / 100.0) < 0.06, (cents, t)
        o = O.analyze(x, 44100, {"enable_key_tuning_compensation": 1}, dump=True, fast=True)
        assert float(o.farray("key.tuning")[0]) == pytest.approx(np.sign(cents) * 0.08, abs=1e-7)
    x = synth.render_progression(7, 12, 44100, tonic=0, minor=False, bpm=120, detune_cents=0.0)
    o = O.analyze(x, 44100, {"enable_key_tuning_compensation": 1, "key_tuning_max_abs_semitones": 0.5}, dump=True, fast=True)
    assert abs(float(o.farray("key.tuning")[0])) < 0.1  # bin-centre quantisation leaves a small bias
