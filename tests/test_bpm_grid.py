"""BPM grids beyond 256 hypotheses: a wider min_bpm..max_bpm range or a finer bpm_resolution.

The grid is the reference's f32 loop `bpm = min_bpm; while bpm <= max_bpm { ..; bpm += bpm_resolution }`
(tempogram_autocorr.rs:79-178, comb_filter.rs:96-215): its count and values come from the accumulation.  Grids of at
most 256 hypotheses keep the per-hypothesis kernels; larger ones take the distinct-lag autocorrelation kernel, the
table lookups of the scoring kernel and the comb filterbank across CTAs.  Above 32768 hypotheses (which includes
every grid whose accumulation stalls) the configuration is rejected with NotImplemented."""
import ctypes as C
import time

import numpy as np
import pytest

import oracle_lib as O
import synth
import stratum_dsp_b200 as S
from gpu_common import assert_parity

SR = 44100
BOUND = 32768
GRIDS = [(40.0, 240.0, 1.0, 201), (40.0, 300.0, 1.0, 261), (40.0, 240.0, 0.5, 401), (40.0, 240.0, 0.1, 2000), (40.0, 240.0, 0.01, 20006),
         (30.0, 300.0, 0.05, None)]


def _grid(lo, hi, res, cap=BOUND + 8):
    L = S.lib()
    L.stratum_b200_debug_bpm_grid.argtypes = [C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_int32]
    L.stratum_b200_debug_bpm_grid.restype = C.c_int32
    out = np.zeros(cap, np.float32)
    n = L.stratum_b200_debug_bpm_grid(lo, hi, res, out.ctypes.data, cap)
    return n, out[:max(n, 0)]


def _numpy_grid(lo, hi, res):
    lo, hi, res = np.float32(lo), np.float32(hi), np.float32(res)
    out, b = [], lo
    while b <= hi:
        out.append(b)
        b = np.float32(b + res)
    return np.array(out, np.float32)


def _oracle_tempogram_bpms(lo, hi, res):
    L = O.lib()
    f32p = C.POINTER(C.c_float)
    L.so_u_tempogram.argtypes = [C.c_int, f32p, C.c_int, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, f32p, f32p, C.c_int]
    nov = np.random.default_rng(5).random(64).astype(np.float32)
    cap = BOUND + 8
    b, v = np.zeros(cap, np.float32), np.zeros(cap, np.float32)
    n = L.so_u_tempogram(1, nov.ctypes.data_as(f32p), nov.size, SR, 512, lo, hi, res, b.ctypes.data_as(f32p), v.ctypes.data_as(f32p), cap)
    assert n > 0
    return np.sort(b[:n])  # the oracle's list is in strength order


@pytest.mark.parametrize("lo,hi,res,count", GRIDS)
def test_grid_is_the_reference_f32_loop(lo, hi, res, count):
    n, got = _grid(lo, hi, res)
    want = _numpy_grid(lo, hi, res)
    assert n == len(want) and np.array_equal(got, want)
    if count is not None:
        assert n == count
    assert np.array_equal(got, _oracle_tempogram_bpms(lo, hi, res))
    assert np.all(np.diff(got) > 0)


def test_fine_grid_drifts_from_index_arithmetic():
    # why the scoring kernel looks hypotheses up by value on fine grids: at 0.01 the accumulated values run 5 steps off min + i * res
    n, got = _grid(40.0, 240.0, 0.01)
    drift = (got.astype(np.float64) - (40.0 + 0.01 * np.arange(n))) / 0.01
    assert n == 20006 and abs(drift[-1]) > 5.0


@pytest.mark.parametrize("lo,hi,res", [(40.0, 240.0, 0.005), (40.0, 240.0, 1e-6)])
def test_grids_beyond_the_bound_are_refused_at_once(lo, hi, res):
    # 40..240 at 0.005 has 39 985 hypotheses; at 1e-6 the accumulation stalls at 40 (the reference's loop never ends)
    t = time.perf_counter()
    n, _ = _grid(lo, hi, res)
    assert n == -1 and time.perf_counter() - t < 1.0


def test_validation_without_a_device():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    x = [np.ones(4096, np.float32)]
    for kw in ({"bpm_resolution": 0.005}, {"bpm_resolution": 1e-6}):
        with pytest.raises(S.AnalysisError) as e:
            S.analyze_batch(x, SR, S.AnalysisConfig(**kw))
        assert e.value.kind == "NotImplemented" and "32768" in e.value.message, kw
    for kw in ({"max_bpm": 300.0}, {"bpm_resolution": 0.01}):  # 261 and 20 006 hypotheses pass validation
        with pytest.raises(S.AnalysisError) as e:
            S.analyze_batch(x, SR, S.AnalysisConfig(**kw))
        assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message, kw


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _tracks():
    # the three tracks of test_gpu_parity.py::test_accepted_config_switches_match_the_oracle; the 76 BPM one escalates
    xs = [synth.render(synth.TrackParams(76.0, 4, 1, 0.4, 0.08, SR, 24 * SR)), synth.render(synth.c2_params(99, 18 * SR, SR))]
    quiet = np.concatenate([np.zeros(SR, np.float32), xs[1][: 10 * SR] * np.float32(0.5), np.zeros(2 * SR, np.float32)])
    return xs + [quiet]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", [
    {"max_bpm": 300.0},
    {"bpm_resolution": 0.5},
    {"bpm_resolution": 0.1},
    {"bpm_resolution": 0.01},
    {"min_bpm": 30.0, "max_bpm": 300.0, "bpm_resolution": 0.05},
    {"bpm_resolution": 0.1, "force_legacy_bpm": 1},                     # the comb filterbank decides
    {"bpm_resolution": 0.1, "enable_bpm_fusion": 1},
    {"bpm_resolution": 0.1, "hop_size": 256},                           # the base path's own slot (SLOT_BASE_ALT)
    {"bpm_resolution": 0.1, "enable_hpss_onsets": 1, "enable_tempogram_percussive_fallback": 1},  # percussive slot
])
def test_fine_grids_match_the_oracle(cfg):
    xs = _tracks()
    res = S.analyze_batch(xs, SR, S.AnalysisConfig(**cfg))
    for i, (x, g) in enumerate(zip(xs, res)):
        assert_parity(g, O.analyze(x, SR, cfg, fast=True), f"{cfg} track {i}")
    assert any(g.metadata.tempogram_multi_res_triggered for g in res) or cfg.get("force_legacy_bpm")


@pytest.mark.gpu
def test_fine_grid_48k_track():
    cfg = {"bpm_resolution": 0.1}
    p = synth.c2_params(41, 20 * 48000, 48000)
    x = synth.render(p)
    assert_parity(S.analyze_audio(x, 48000, S.AnalysisConfig(**cfg)), O.analyze(x, 48000, cfg, fast=True), "48 kHz")


@pytest.mark.gpu
def test_fine_grid_tempogram_candidates():
    # compared as in test_gpu_parity.py::test_tempogram_candidates_metadata
    cfg = {"bpm_resolution": 0.1, "emit_tempogram_candidates": 1}
    for bpm in (74.0, 121.0):
        x = synth.render(synth.TrackParams(bpm, 2, 0, 0.25, 0.1, SR, 20 * SR))
        o = O.analyze(x, SR, cfg, fast=True)
        g = S.analyze_audio(x, SR, S.AnalysisConfig(**cfg))
        assert_parity(g, o, f"{cfg} bpm={bpm}")
        exp = o.farray("result.candidates").reshape(-1, 5)
        got = g.metadata.tempogram_candidates
        assert got is not None and len(got) == len(exp)
        for (b, sc, fn, an, sel), e in zip(got, exp):
            assert b == e[0] and abs(sc - e[1]) <= 1e-3 * max(abs(e[1]), 1e-6) + 1e-6 and bool(e[4]) == sel
            assert abs(fn - e[2]) < 1e-3 and abs(an - e[3]) < 1e-3


def _dumps(x, cfg):
    S.debug_enable(True)
    try:
        g = S.analyze_audio(x, SR, S.AnalysisConfig(**cfg))
        return g, {k: S.debug_array(k) for k in ("base.tg.ac.full", "h256.tg.ac.full", "h1024.tg.ac.full", "legacy.comb_raw")}
    finally:
        S.debug_enable(False)


@pytest.mark.gpu
def test_new_kernels_are_bit_identical_to_the_per_hypothesis_kernels():
    # 40..240 at 0.5 (401 hypotheses: distinct-lag tempogram, comb filterbank across CTAs) holds the integer BPMs of the
    # 1.0 grid (201: the per-hypothesis kernels) at its even entries, exactly: both sets of kernels must give the same bits there
    x = _tracks()[0]
    g1, d1 = _dumps(x, {})
    g2, d2 = _dumps(x, {"bpm_resolution": 0.5})
    assert g1.metadata.tempogram_multi_res_triggered and g2.metadata.tempogram_multi_res_triggered
    for k in d1:
        a, b = d1[k], d2[k]
        assert a is not None and b is not None, k
        assert a.size == 201 and b.size == 401, (k, a.size, b.size)
        assert np.array_equal(b[::2].view(np.uint32), a.view(np.uint32)), k
    o = O.analyze(x, SR, {"bpm_resolution": 0.5}, dump=True)
    assert np.array_equal(d2["legacy.comb_raw"], o.farray("legacy.comb.raw"))  # integer onset positions: exact


@pytest.mark.gpu
def test_fine_grid_batches_match_single_calls(monkeypatch):
    cfg = S.AnalysisConfig(bpm_resolution=0.1)
    tracks, srs = [], []
    for i in range(6):
        p = synth.c5_params(i)
        p.n_samples = min(p.n_samples, 30 * p.sample_rate)
        tracks.append(synth.render(p))
        srs.append(p.sample_rate)
    a = S.analyze_batch(tracks, srs, cfg)
    monkeypatch.setenv("STRATUM_B200_WAVE_MAX_TRACKS", "2")
    b = S.analyze_batch(tracks, srs, cfg)
    monkeypatch.delenv("STRATUM_B200_WAVE_MAX_TRACKS")
    for x, sr, u, v in zip(tracks, srs, a, b):
        s = S.analyze_audio(x, sr, cfg)
        for w in (v, s):
            assert u.bpm == w.bpm and u.bpm_confidence == w.bpm_confidence and u.key == w.key
            assert np.array_equal(u.beat_grid.beats, w.beat_grid.beats)
