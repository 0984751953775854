"""BS.1770-4 / EBU R128 loudness (stratum_b200_loudness_batch_pcm): the host-side filters and call validation on the CPU; on the
GPU, parity with the float64 reference in loudness_ref.py, the EBU Tech 3341 / 3342 style analytic cases, and bit-identical
results across batching, upload chunks, the device entry and sharding."""
import ctypes as C
import math
import os
import re
from pathlib import Path

import numpy as np
import pytest

import loudness_ref as R
import stratum_dsp_b200 as S
import synth

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()
FIELDS = ("integrated_lufs", "momentary_max_lufs", "short_term_max_lufs", "loudness_range_lu", "sample_peak", "true_peak", "n_momentary",
          "n_short_term", "sample_rate", "channels", "frames")


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_loudness_symbols_declared_and_exported():
    L = S.lib()
    for s in ("stratum_b200_loudness_batch_pcm", "stratum_b200_loudness_batch_pcm_device", "stratum_b200_debug_loudness_filters"):
        assert re.search(rf"\b{s}\s*\(", HEADER), s
        assert hasattr(L, s), s
    assert "typedef struct StratumLoudness" in HEADER


def test_loudness_struct_size():
    assert S.lib().stratum_b200_sizeof(3) == C.sizeof(S.StratumLoudness)
    assert S.lib().stratum_b200_sizeof(4) == 0


def test_kweighting_48k_equals_published_tables():
    k, _, L = S.loudness_filters(48000)
    assert L == 4
    pub = [1.53512485958697, -2.69169618940638, 1.19839281085285, -1.69065929318241, 0.73248077421585, 1.0, -2.0, 1.0,
           -1.99004745483398, 0.99007225036621]
    assert np.max(np.abs(k - np.array(pub))) < 1e-9


@pytest.mark.parametrize("sr", [8000, 22050, 44100, 96000, 192000, 384000])
def test_kweighting_matches_float64_reference(sr):
    k, _, _ = S.loudness_filters(sr)
    (b1, a1), (b2, a2) = R.kweight(sr)
    ref = np.concatenate([b1, a1[1:], b2, a2[1:]])
    np.testing.assert_allclose(k, ref, rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("sr,L", [(44100, 4), (48000, 4), (95999, 4), (96000, 2), (191999, 2), (192000, 1), (384000, 1)])
def test_true_peak_taps_are_symmetric_and_interpolating(sr, L):
    _, t, got = S.loudness_filters(sr)
    assert got == L
    assert np.array_equal(t, t[::-1])
    assert t[24] == 1.0
    for k in range(1, 24 // L + 1):
        assert t[24 + L * k] == 0.0 and t[24 - L * k] == 0.0
    np.testing.assert_allclose(t, R.taps(L).astype(np.float32), rtol=0, atol=0)


@pytest.mark.parametrize("sr", [0, 7999, 384001])
def test_filters_reject_sample_rates_outside_the_range(sr):
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_filters(sr)
    assert e.value.kind == "NotImplemented" and "8000..384000" in e.value.message


def test_loudness_has_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    t = R.encode(np.zeros((48000, 2)), S.PCM_S16, 48000)
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_batch_pcm([t])
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message
    with pytest.raises(S.AnalysisError) as e:  # the address is never dereferenced: the call stops at the device lookup
        S.loudness_batch_pcm_device(1 << 20, np.array([0, t.data.size], np.uint64), [48000], [2], [S.PCM_S16])
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message


def _raw_call(data, offsets, srs, chans, fmts):
    n = len(offsets) - 1
    off = np.ascontiguousarray(offsets, np.uint64)
    arr = lambda v: np.ascontiguousarray(v, np.uint32)
    s, c, f = arr(srs), arr(chans), arr(fmts)
    res = (S.StratumLoudness * max(n, 1))()
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint32))
    return S.lib().stratum_b200_loudness_batch_pcm(data.ctypes.data if data is not None else None, off.ctypes.data_as(C.POINTER(C.c_uint64)), p(s), p(c),
                                                    p(f), n, None, 0, res)


@pytest.mark.parametrize("case", ["unknown_format", "zero_channels", "too_many_channels", "partial_frame", "null_pcm"])
def test_malformed_calls_are_rejected_whole(case):
    data = np.zeros(4 * 100, np.uint8)
    offsets, srs, chans, fmts = [0, 200, 400], [48000, 48000], [2, 2], [S.PCM_S16, S.PCM_S16]
    if case == "unknown_format":
        fmts = [S.PCM_S16, 9]
    elif case == "zero_channels":
        chans = [2, 0]
    elif case == "too_many_channels":
        chans = [2, 65]
    elif case == "partial_frame":
        offsets = [0, 200, 399]
    else:
        data = None
    assert _raw_call(data, offsets, srs, chans, fmts) == S.INVALID_INPUT
    assert S.last_error()


# ---- GPU: parity with the float64 reference ----------------------------------------------------------------------------
def _check(g: S.Loudness, ref: dict, label=""):
    assert g.error is None, f"{label}: {g.error}"
    assert g.n_momentary == ref["n_momentary"] and g.n_short_term == ref["n_short_term"], label
    for f, tol in (("integrated_lufs", 0.01), ("momentary_max_lufs", 0.01), ("short_term_max_lufs", 0.01), ("loudness_range_lu", 0.02)):
        a, b = getattr(g, f), ref[f]
        if math.isinf(b):
            assert a == b, f"{label} {f}: {a} vs {b}"
        else:
            assert abs(a - b) <= tol, f"{label} {f}: {a} vs {b}"
    assert g.sample_peak == ref["sample_peak"], f"{label} sample_peak: {g.sample_peak} vs {ref['sample_peak']}"
    if "true_peak" in ref:
        assert abs(g.true_peak - ref["true_peak"]) <= 1e-5 * ref["true_peak"], f"{label} true_peak: {g.true_peak} vs {ref['true_peak']}"


def _stereo_c2(i, n, sr):
    return np.stack([synth.render(synth.c2_params(i, n, sr)), synth.render(synth.c2_params(i + 1000, n, sr))], axis=1)


def _multichannel(C, n, sr, seed):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / sr
    cols = []
    for c in range(C):
        f = 40.0 + 5000.0 * rng.random()
        env = 0.2 + 0.8 * (0.5 + 0.5 * np.sin(2 * np.pi * t / (1.0 + 3 * rng.random())))
        cols.append(0.3 * env * np.sin(2 * np.pi * f * t) + 0.05 * rng.standard_normal(n))
    return np.clip(np.stack(cols, axis=1), -1.0, 1.0)


@pytest.mark.gpu
def test_parity_c2_stereo_three_minutes():
    tracks = [R.encode(_stereo_c2(i, 7_938_000, 44100), S.PCM_S16, 44100) for i in range(2)]
    for i, (g, t) in enumerate(zip(S.loudness_batch_pcm(tracks), tracks)):
        _check(g, R.measure(t), f"c2 {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [8000, 22050, 44100, 48000, 96000, 192000])
def test_parity_formats_channels_lengths(sr):
    Sb = (sr + 5) // 10
    lengths = [int(0.3 * sr), 4 * Sb, int(2.9 * sr), 30 * Sb, 20 * sr]
    fmts = [S.PCM_U8, S.PCM_S16, S.PCM_S24, S.PCM_S32, S.PCM_F32, S.PCM_F64]
    chans = [1, 2, 6, 8, 5, 4]
    tracks = []
    for i, n in enumerate(lengths):
        for j in range(2):
            q = (i * 2 + j) % len(fmts)
            tracks.append(R.encode(_multichannel(chans[(i + 3 * j) % len(chans)], n, sr, 100 * i + j), fmts[q], sr))
    got = S.loudness_batch_pcm(tracks)
    for k, (g, t) in enumerate(zip(got, tracks)):
        _check(g, R.measure(t), f"sr {sr} track {k} fmt {t.fmt} C {t.channels} frames {t.frames}")


@pytest.mark.gpu
def test_parity_c4_sixty_minute_mix():
    x = synth.c4_mix()
    t = R.encode(x, S.PCM_F32, 44100)
    del x
    (g,) = S.loudness_batch_pcm([t])
    _check(g, R.measure(t), "c4")


# ---- GPU: analytic cases (EBU Tech 3341 / 3342 style, 48 kHz) ---------------------------------------------------------------
SR = 48000


def _sine(db, seconds, f=1000.0, channels=2, phase0=0.0):
    n = int(seconds * SR)
    a = 10.0 ** (db / 20.0)
    x = a * np.sin(2 * np.pi * f * np.arange(n) / SR + phase0)
    return np.repeat(x[:, None], channels, axis=1)


def _one(x, fmt=S.PCM_F32):
    (g,) = S.loudness_batch_pcm([R.encode(x, fmt, SR)])
    assert g.error is None
    return g


@pytest.mark.gpu
@pytest.mark.parametrize("db", [-23.0, -33.0])
def test_stereo_sine_reads_its_level(db):
    g = _one(_sine(db, 20.0))
    for v in (g.integrated_lufs, g.momentary_max_lufs, g.short_term_max_lufs):
        assert abs(v - db) <= 0.1, (db, g)


@pytest.mark.gpu
@pytest.mark.parametrize("levels,durs", [((-36, -23, -36), (10, 60, 10)), ((-72, -36, -23, -36, -72), (10, 10, 60, 10, 10))])
def test_gates(levels, durs):
    g = _one(np.concatenate([_sine(l, d) for l, d in zip(levels, durs)]))
    assert abs(g.integrated_lufs + 23.0) <= 0.1, g


@pytest.mark.gpu
@pytest.mark.parametrize("levels,lra", [((-20, -30), 10.0), ((-20, -15), 5.0), ((-40, -20), 20.0), ((-50, -35, -20, -35, -50), 15.0)])
def test_loudness_range(levels, lra):
    g = _one(np.concatenate([_sine(l, 20.0) for l in levels]))
    assert abs(g.loudness_range_lu - lra) <= 0.1, g


@pytest.mark.gpu
@pytest.mark.parametrize("C,ch,expect", [(2, 0, -3.01), (6, 4, -1.52), (6, 3, -math.inf)])
def test_channel_weights(C, ch, expect):
    x = np.zeros((20 * SR, C))
    x[:, ch] = np.sin(2 * np.pi * 997.0 * np.arange(20 * SR) / SR)
    g = _one(x)
    if math.isinf(expect):
        assert g.integrated_lufs == -math.inf
    else:
        assert abs(g.integrated_lufs - expect) <= 0.05, g


@pytest.mark.gpu
def test_true_peak_of_quarter_rate_sine():
    A = 0.5
    n = np.arange(10 * SR)
    x = A * np.sin(np.pi * n / 2 + np.pi / 4)
    g = _one(np.stack([x, x], axis=1), S.PCM_F64)
    assert abs(g.sample_peak - A * 0.7071) < 1e-4
    db = 20 * math.log10(g.true_peak / A)
    assert -0.4 <= db <= 0.2, db


# ---- GPU: invariance and per-track failures ----------------------------------------------------------------------------------
def _fields(g: S.Loudness):
    return tuple(getattr(g, f) for f in FIELDS)


@pytest.mark.gpu
def test_results_do_not_depend_on_batch_chunks_entry_or_devices(monkeypatch):
    import torch

    sr = 44100
    probe = R.encode(_stereo_c2(3, 30 * sr, sr), S.PCM_S16, sr)
    others = [R.encode(_multichannel(c, n, r, 7 + c), f, r) for c, n, r, f in
              ((1, 5 * sr, sr, S.PCM_S24), (6, 12 * 48000, 48000, S.PCM_F32), (2, 3 * 96000, 96000, S.PCM_S16), (8, 40 * sr, sr, S.PCM_U8))]
    alone = _fields(S.loudness_batch_pcm([probe])[0])
    batch = others[:2] + [probe] + others[2:]
    assert _fields(S.loudness_batch_pcm(batch)[2]) == alone
    assert _fields(S.loudness_batch_pcm(batch, devices=[0, 0])[2]) == alone
    # chunks of 1 MB of mono f32 frames: every track lands in a chunk of its own, and the batch spans several staging rounds
    monkeypatch.setenv("STRATUM_B200_STAGE_MB", "1")
    split = S.loudness_batch_pcm(batch)
    monkeypatch.delenv("STRATUM_B200_STAGE_MB")
    assert _fields(split[2]) == alone
    whole = S.loudness_batch_pcm(batch)
    assert [_fields(g) for g in split] == [_fields(g) for g in whole]
    cat = np.concatenate([t.data for t in batch])
    offsets = np.zeros(len(batch) + 1, np.uint64)
    offsets[1:] = np.cumsum([t.data.size for t in batch])
    d = torch.from_numpy(cat).cuda()
    dev = S.loudness_batch_pcm_device(d.data_ptr(), offsets, [t.sample_rate for t in batch], [t.channels for t in batch], [t.fmt for t in batch],
                                      device=d.device.index)
    torch.cuda.synchronize()
    assert [_fields(g) for g in dev] == [_fields(g) for g in whole]


@pytest.mark.gpu
def test_failing_tracks_fail_alone():
    sr = 48000
    good = R.encode(_multichannel(2, 5 * sr, sr, 3), S.PCM_S16, sr)
    empty = S.PcmTrack(np.zeros(0, np.uint8), S.PCM_S16, 2, sr)
    zero_sr = S.PcmTrack(good.data.copy(), S.PCM_S16, 2, 0)
    low = S.PcmTrack(good.data.copy(), S.PCM_S16, 2, 7999)
    high = S.PcmTrack(good.data.copy(), S.PCM_S16, 2, 400000)
    got = S.loudness_batch_pcm([good, empty, zero_sr, good, low, high])
    alone = _fields(S.loudness_batch_pcm([good])[0])
    assert got[0].error is None and got[3].error is None
    assert _fields(got[0]) == alone and _fields(got[3]) == alone
    assert got[1].error.kind == "InvalidInput" and got[2].error.kind == "InvalidInput"
    for g in (got[4], got[5]):
        assert g.error.kind == "NotImplemented" and "8000..384000" in g.error.message
