"""frame_size 4096 and 8192 on the tempo path.

A larger analysis frame widens every STFT bin's share of the bass: at 44.1 kHz the low tempogram band of a 2048-point frame spans
bins 1..8, of a 4096-point frame twice and of an 8192-point frame four times as many.  The frame size reaches the silence
detector (frame F, hop F/2), the energy-flux frames, the tempo-path STFT at hops 512 / 256 / 1024, the feature kernels and HPSS
(F/2 + 1 bins), the band edges and mel filterbank, and, with enable_key_stft_override off, the key STFT.  2048 keeps its kernels;
smaller sizes, 16384 and above and non-powers of two are rejected with NotImplemented."""
import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle_lib as O
import synth
import stratum_dsp_b200 as S
from gpu_common import assert_parity

SR = 44100
T3 = 7_938_000  # 3 minutes at 44.1 kHz
SIZES = [4096, 8192]


def test_validation_without_a_device():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    x = [np.ones(4096, np.float32)]
    for f in SIZES:
        with pytest.raises(S.AnalysisError) as e:
            S.analyze_batch(x, SR, S.AnalysisConfig(frame_size=f))
        assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message, f
    for f in (512, 1024, 3000, 16384):
        with pytest.raises(S.AnalysisError) as e:
            S.analyze_batch(x, SR, S.AnalysisConfig(frame_size=f))
        assert e.value.kind == "NotImplemented" and "2048, 4096 or 8192" in e.value.message, f


def _plan(lens, budget_gb, cfg):
    L = S.lib()
    L.stratum_b200_debug_plan_waves.restype = C.c_uint32
    n = len(lens)
    off = np.zeros(n + 1, np.uint64)
    off[1:] = np.cumsum(np.asarray(lens, np.uint64))
    sr = np.full(n, SR, np.uint32)
    out = np.zeros(n, np.uint32)
    nw = L.stratum_b200_debug_plan_waves(off.ctypes.data_as(C.POINTER(C.c_uint64)), sr.ctypes.data_as(C.POINTER(C.c_uint32)), n,
                                         C.byref(cfg._c), C.c_double(budget_gb), out.ctypes.data_as(C.POINTER(C.c_uint32)))
    return nw, out


def test_wave_planner_sizes_spectrograms_by_bins():
    # a three-minute track's hop-512 spectrogram is 64 MB at 2048 and 254 MB at 8192: the same budget holds fewer tracks per wave
    nw = {}
    for f in (2048, 4096, 8192):
        nw[f], w = _plan([T3] * 200, 20.0, S.AnalysisConfig(frame_size=f))
        assert np.all(np.diff(w) >= 0) and w[0] == 0 and w[-1] == nw[f] - 1, f  # contiguous, in order, every track placed
    assert nw[8192] > nw[2048] and nw[4096] >= nw[2048]
    n, _ = _plan([20 * T3], 20.0, S.AnalysisConfig(frame_size=8192))  # one 60-minute mix still plans
    assert n == 1


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def _tracks():
    # the three tracks of test_bpm_grid.py; the 76 BPM one escalates
    xs = [synth.render(synth.TrackParams(76.0, 4, 1, 0.4, 0.08, SR, 24 * SR)), synth.render(synth.c2_params(99, 18 * SR, SR))]
    quiet = np.concatenate([np.zeros(SR, np.float32), xs[1][: 10 * SR] * np.float32(0.5), np.zeros(2 * SR, np.float32)])
    return xs + [quiet]


CONFIGS = [
    {},
    {"hop_size": 256},
    {"hop_size": 1024},
    {"hop_size": 400},                                                      # unaligned frame starts, generic frame RMS
    {"enable_hpss_onsets": 1, "enable_tempogram_percussive_fallback": 1},  # percussive slot
    {"tempogram_band_seed_only": 0, "enable_tempogram_mel_novelty": 1},
    {"force_legacy_bpm": 1},
    {"enable_key_stft_override": 0},                                        # the key STFT at frame_size / hop_size
]


@pytest.mark.gpu
@pytest.mark.parametrize("frame", SIZES)
@pytest.mark.parametrize("cfg", CONFIGS)
def test_frame_sizes_match_the_oracle(frame, cfg):
    cfg = dict(cfg, frame_size=frame)
    xs = _tracks()
    res = S.analyze_batch(xs, SR, S.AnalysisConfig(**cfg))
    with ThreadPoolExecutor(len(xs)) as ex:  # the oracle's HPSS at 8192 points takes minutes per track; its calls release the GIL
        want = list(ex.map(lambda x: O.analyze(x, SR, cfg, fast=True), xs))
    for i, (g, o) in enumerate(zip(res, want)):
        assert_parity(g, o, f"{cfg} track {i}")
    assert any(g.metadata.tempogram_multi_res_triggered for g in res) or cfg.get("force_legacy_bpm")


@pytest.mark.gpu
@pytest.mark.parametrize("frame", SIZES)
def test_48k_track(frame):
    cfg = {"frame_size": frame}
    x = synth.render(synth.c2_params(41, 20 * 48000, 48000))
    assert_parity(S.analyze_audio(x, 48000, S.AnalysisConfig(**cfg)), O.analyze(x, 48000, cfg, fast=True), f"48 kHz {frame}")


@pytest.mark.gpu
@pytest.mark.parametrize("frame", SIZES)
def test_tracks_shorter_than_the_frame(frame):
    # below 2048 samples: one short silence frame; between 2048 and F: no STFT frame and no key frame at all
    cfg = {"frame_size": frame}
    rng = np.random.default_rng(7)
    for n in (1500, 2047, 3000, frame - 1, frame, frame + 3000):
        x = (rng.standard_normal(n) * 0.2).astype(np.float32)
        o = O.analyze(x, SR, cfg)
        try:
            g = S.analyze_audio(x, SR, S.AnalysisConfig(**cfg))
        except S.AnalysisError as e:
            assert o.status == e.code, (n, e, o.error)
            continue
        assert_parity(g, o, f"noise n={n} frame={frame}")


@pytest.mark.gpu
@pytest.mark.parametrize("frame", SIZES)
def test_spectrograms_are_bit_identical(frame):
    x = synth.render(synth.c2_params(95, 7 * SR, SR))
    cfg = {"frame_size": frame, "enable_hpss_onsets": 1}
    o = O.analyze(x, SR, cfg, dump=True, fast=True)
    S.debug_enable(True)
    try:
        g = S.analyze_audio(x, SR, S.AnalysisConfig(**cfg))
        gain = np.float32(S.debug_array("gain")[0])
        y = (x[g.trim_start:g.trim_end] * gain).astype(np.float32)
        want = O.stft(y, frame, 512)[:64].ravel()
        got = S.debug_array("spec512_head")
        assert got.size == want.size == 64 * (frame // 2 + 1)
        assert np.array_equal(got, want)
        ph = o.farray("hpss.perc_head")
        assert ph.size == want.size and np.array_equal(S.debug_array("hpss.perc_head")[: ph.size], ph)
        assert np.array_equal(S.debug_array("onset.spectral_flux"), o.farray("onset.spectral_flux"))
    finally:
        S.debug_enable(False)
    assert_parity(g, o, f"dumps {frame}")


KEY_DUMPS = ("key.hpcp_raw", "key.hpcp_smooth", "key.energy", "key.weights", "key.seg_scores", "key.band_head")


def _key_run(x, cfg):
    S.debug_enable(True)
    try:
        g = S.analyze_audio(x, SR, S.AnalysisConfig(**cfg))
        return g, {k: S.debug_array(k) for k in KEY_DUMPS}
    finally:
        S.debug_enable(False)


@pytest.mark.gpu
def test_key_geometry_at_8192_equals_the_default():
    # frame_size 8192, hop 512 with the override off is the default key geometry (8192 / 512): the key path must not notice
    x = _tracks()[1]
    g0, d0 = _key_run(x, {})
    g1, d1 = _key_run(x, {"frame_size": 8192, "enable_key_stft_override": 0})
    assert (g1.trim_start, g1.trim_end) == (g0.trim_start, g0.trim_end)  # same samples reach the key path
    assert g1.key == g0.key and g1.key_confidence == g0.key_confidence and g1.key_clarity == g0.key_clarity
    for k in KEY_DUMPS:
        a, b = d0[k], d1[k]
        assert a is not None and b is not None and a.size == b.size, k
        if k == "key.seg_scores":
            # 24 scores per row: the segment windows, then the whole-track row (scored only when voting rejects every window) and one
            # spare row; those two are arena capacity that this track never writes
            a, b = a[:-48], b[:-48]
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), k


@pytest.mark.gpu
@pytest.mark.parametrize("frame", SIZES)
def test_batches_match_single_calls(frame, monkeypatch):
    cfg = S.AnalysisConfig(frame_size=frame)
    tracks, srs = [], []
    for i in range(6):
        p = synth.c5_params(i)
        p.n_samples = min(p.n_samples, 30 * p.sample_rate)
        tracks.append(synth.render(p))
        srs.append(p.sample_rate)
    assert {44100, 48000} <= set(srs)
    a = S.analyze_batch(tracks, srs, cfg)
    monkeypatch.setenv("STRATUM_B200_WAVE_MAX_TRACKS", "2")
    b = S.analyze_batch(tracks, srs, cfg)
    monkeypatch.delenv("STRATUM_B200_WAVE_MAX_TRACKS")
    for x, sr, u, v in zip(tracks, srs, a, b):
        s = S.analyze_audio(x, sr, cfg)
        for w in (v, s):
            assert u.bpm == w.bpm and u.bpm_confidence == w.bpm_confidence and u.key == w.key and u.key_clarity == w.key_clarity
            assert np.array_equal(u.beat_grid.beats, w.beat_grid.beats) and np.array_equal(u.onsets, w.onsets)
