"""Loudness series (stratum_b200_loudness_series_pcm, its device and combined forms, stratum_b200_loudness_series_lengths): the lengths
rule, declarations, Python keywords and layout on the CPU; on the GPU, the series against the float64 reference of
loudness_series_ref.py, the maxima invariants, NULL and partial requests, invariance across entries, chunks and devices, channel maps,
EBU Tech 3341 signals, and the launches and read-backs."""
import ctypes as C
import inspect
import math
import re
from pathlib import Path

import numpy as np
import pytest

import loudness_ref as R
import loudness_series_ref as RS
import stratum_dsp_b200 as S
from test_loudness import _multichannel
from test_loudness_layout import FMTS, LOUD_OUT_BYTES, _all, _batch, _full

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()
U8P, U32P, U64P, F64P = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_double)
SERIES = ("momentary_lufs", "short_term_lufs", "sample_peak", "true_peak")
ENTRIES = ("stratum_b200_loudness_series_pcm", "stratum_b200_loudness_series_pcm_device", "stratum_b200_analyze_loudness_series_pcm",
           "stratum_b200_loudness_series_lengths")


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_symbols_declared_and_exported():
    L = S.lib()
    for s in ENTRIES:
        assert re.search(rf"\b{s}\s*\(", HEADER), s
        assert hasattr(L, s), s


def _lengths_by_definition(sr, frames):
    if frames == 0 or sr == 0 or sr < 8000 or sr > 384000:
        return 0, 0, 0
    Sb = (sr + 5) // 10
    nfull = frames // Sb
    return max(0, nfull - 3), max(0, nfull - 29), -(-frames // Sb)


@pytest.mark.parametrize("sr", [0, 7999, 8000, 44100, 48000, 384000, 384001])
def test_series_lengths_follow_the_definition(sr):
    Sb = max((sr + 5) // 10, 1)
    L = S.lib()
    for frames in (0, 1, Sb - 1, 4 * Sb - 1, 4 * Sb, 30 * Sb + 7, 10 ** 7 + 3):
        n = (C.c_uint32 * 3)(7, 7, 7)
        st = L.stratum_b200_loudness_series_lengths(sr, frames, C.cast(C.byref(n, 0), U32P), C.cast(C.byref(n, 4), U32P), C.cast(C.byref(n, 8), U32P))
        want = _lengths_by_definition(sr, frames)
        assert tuple(n) == want, (sr, frames)
        assert S.loudness_series_lengths(sr, frames) == want
        if frames == 0 or sr == 0:
            assert st == S.INVALID_INPUT
        elif sr < 8000 or sr > 384000:
            assert st == S.NOT_IMPLEMENTED
        else:
            assert st == S.OK
        assert L.stratum_b200_loudness_series_lengths(sr, frames, None, None, None) == st  # every pointer may be NULL


def test_python_keyword_and_layout():
    for fn in (S.loudness_batch_pcm, S.loudness_batch_pcm_device, S.loudness_albums_pcm, S.loudness_albums_pcm_device, S.analyze_loudness_pcm):
        p = inspect.signature(fn).parameters["series"]
        assert p.kind == p.KEYWORD_ONLY and p.default is False, fn.__name__
    assert S.Loudness(0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0, 0, 0, 0, 0).series is None
    sr = 48000
    tracks = [R.encode(np.zeros((n, c)), f, r) for n, c, f, r in ((4 * 4800, 2, S.PCM_S16, sr), (0, 3, S.PCM_S24, sr), (31 * 4410 + 5, 1, S.PCM_F64, 44100),
                                                                    (9000, 2, S.PCM_U8, 7999))]
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    lengths, arrays = S._series_args(True, offsets, srs, chans, fmts)
    assert lengths == [(1, 0, 4), (0, 0, 0), (28, 2, 32), (0, 0, 0)]
    assert [a.size for a in arrays] == [29, 2, 36, 36] and all(a.dtype == np.float64 for a in arrays)
    assert S._series_args(False, offsets, srs, chans, fmts) == (None, [None] * 4)
    # the split hands each track its own slice, in track order
    arrays = [np.arange(a.size, dtype=np.float64) + 1000 * k for k, a in enumerate(arrays)]
    loud = [S.Loudness(0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0, 0, r, c, 0, None if ln[2] else S.AnalysisError(1, "x")) for r, c, ln in
            zip((sr, sr, 44100, 7999), (2, 3, 1, 2), lengths)]
    S._with_series(loud, lengths, arrays)
    assert list(loud[2].series.momentary_lufs) == list(range(1, 29)) and list(loud[2].series.sample_peak) == [2000.0 + v for v in range(4, 36)]
    assert list(loud[2].series.true_peak) == [3000.0 + v for v in range(4, 36)] and list(loud[2].series.short_term_lufs) == [1000.0, 1001.0]
    assert loud[0].series.step_seconds == 0.1 and loud[2].series.step_seconds == 4410 / 44100
    assert loud[1].series.sample_peak.size == 0 and loud[1].series.step_seconds == 0.0


def test_series_entries_have_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    t = R.encode(np.zeros((48000, 2)), S.PCM_S16, 48000)
    for call in (lambda: S.loudness_batch_pcm([t], series=True), lambda: S.loudness_albums_pcm([t], [0], series=True),
                 lambda: S.loudness_batch_pcm_device(1 << 20, np.array([0, t.data.size], np.uint64), [48000], [2], [S.PCM_S16], series=True)):
        with pytest.raises(S.AnalysisError) as e:
            call()
        assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message
    with pytest.raises(S.AnalysisError) as e:
        S.analyze_loudness_pcm([t], series=True)
    assert "no CPU fallback" in e.value.message


# ---- GPU -----------------------------------------------------------------------------------------------------------------
def _ser(g):
    return None if g.series is None else (tuple(getattr(g.series, k).tobytes() for k in SERIES), g.series.step_seconds)


def _check_series(g, t, codes=None, label=""):
    ref = RS.series(t, codes)
    for k in ("momentary_lufs", "short_term_lufs"):
        a, b = getattr(g.series, k), ref[k]
        assert a.shape == b.shape, (label, k)
        assert np.array_equal(np.isinf(a), np.isinf(b)) and np.array_equal(a[np.isinf(a)], b[np.isinf(b)]), (label, k)
        f = ~np.isinf(b)
        assert np.all(np.abs(a[f] - b[f]) <= 0.01), (label, k, float(np.max(np.abs(a[f] - b[f]))))
    assert np.array_equal(g.series.sample_peak, ref["sample_peak"]), label
    assert g.series.true_peak.shape == ref["true_peak"].shape, label
    assert np.all(np.abs(g.series.true_peak - ref["true_peak"]) <= 1e-5 * ref["true_peak"]), label


def _check_maxima(g, label=""):
    s = g.series
    assert g.momentary_max_lufs == (s.momentary_lufs.max() if s.momentary_lufs.size else -math.inf), label
    assert g.short_term_max_lufs == (s.short_term_lufs.max() if s.short_term_lufs.size else -math.inf), label
    assert g.sample_peak == s.sample_peak.max() and g.true_peak == s.true_peak.max(), label


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [8000, 44100, 96000, 192000])
def test_series_match_the_float64_reference(sr):
    tracks = _batch(sr)
    got = S.loudness_batch_pcm(tracks, series=True)
    Sb = (sr + 5) // 10
    for i, (g, t) in enumerate(zip(got, tracks)):
        if g.error is not None:  # the 7999 Hz and the empty track
            assert all(getattr(g.series, k).size == 0 for k in SERIES), i
            continue
        n_m, n_q, n_p = S.loudness_series_lengths(sr, t.frames)
        assert (g.series.momentary_lufs.size, g.series.short_term_lufs.size, g.series.sample_peak.size, g.series.true_peak.size) == (n_m, n_q, n_p, n_p)
        assert (n_m, n_q) == (g.n_momentary, g.n_short_term)
        assert g.series.step_seconds == Sb / sr
        _check_series(g, t, label=f"track {i} @ {sr}")
        _check_maxima(g, f"track {i} @ {sr}")
    assert sum(g.error is not None for g in got) == 2


@pytest.mark.gpu
def test_album_maxima_are_the_maxima_over_the_members_entries():
    sr = 44100
    tracks = [R.encode(_multichannel(1 + i % 4, int((4 + 7 * i) * sr), sr, 70 + i), FMTS[i % len(FMTS)], sr) for i in range(6)]
    ids = [0, 1, 0, 1, None, 0]
    got, albums = S.loudness_albums_pcm(tracks, ids, series=True)
    assert all(a.series is None for a in albums)
    for a, alb in enumerate(albums):
        members = [got[i] for i in range(len(tracks)) if ids[i] == a]
        for g in members:
            _check_maxima(g)
        assert alb.momentary_max_lufs == max(g.series.momentary_lufs.max() for g in members if g.series.momentary_lufs.size)
        assert alb.short_term_max_lufs == max((g.series.short_term_lufs.max() for g in members if g.series.short_term_lufs.size), default=-math.inf)
        assert alb.sample_peak == max(g.series.sample_peak.max() for g in members)
        assert alb.true_peak == max(g.series.true_peak.max() for g in members)


def _raw_series(tracks, which, ids=None, n_albums=0, cmap=None):
    """stratum_b200_loudness_series_pcm with the series in `which` (indices into SERIES) requested; returns (status, results, albums,
    arrays with None for the ones not requested)."""
    cat = np.concatenate([t.data for t in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    _, arrays = S._series_args(True, offsets, srs, chans, fmts)
    arrays = [a if k in which else None for k, a in enumerate(arrays)]
    n = len(tracks)
    res, alb = (S.StratumLoudness * n)(), (S.StratumLoudness * max(n_albums, 1))()
    idv = np.array([S.NO_ALBUM if a is None else a for a in ids], np.uint32) if ids is not None else None
    m = np.ascontiguousarray(cmap, np.uint8) if cmap is not None else None
    st = S.lib().stratum_b200_loudness_series_pcm(cat.ctypes.data, offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P), chans.ctypes.data_as(U32P),
                                                  fmts.ctypes.data_as(U32P), n, idv.ctypes.data_as(U32P) if idv is not None else None, n_albums,
                                                  m.ctypes.data_as(U8P) if m is not None else None, None, 0, res, alb, None,
                                                  *[a.ctypes.data_as(F64P) if a is not None else None for a in arrays])
    return st, [_full(S._loudness(r)) for r in res], [_full(S._loudness(alb[a])) for a in range(n_albums)], arrays


@pytest.mark.gpu
def test_null_series_equal_the_mapped_entries_and_subsets_equal_all_four():
    tracks = _batch(48000)
    ids = [i % 3 if i % 4 else None for i in range(len(tracks))]
    cat = np.concatenate([t.data for t in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    n, na = len(tracks), 3
    res, alb = (S.StratumLoudness * n)(), (S.StratumLoudness * na)()
    idv = np.array([S.NO_ALBUM if a is None else a for a in ids], np.uint32)
    assert S.lib().stratum_b200_loudness_mapped_pcm(cat.ctypes.data, offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P), chans.ctypes.data_as(U32P),
                                                    fmts.ctypes.data_as(U32P), n, idv.ctypes.data_as(U32P), na, None, None, 0, res, alb, None) == S.OK
    mapped = ([_full(S._loudness(r)) for r in res], [_full(S._loudness(a)) for a in alb])
    st, t0, a0, _ = _raw_series(tracks, (), ids, na)
    assert st == S.OK and (t0, a0) == mapped
    st, t4, a4, full = _raw_series(tracks, (0, 1, 2, 3), ids, na)
    assert st == S.OK and (t4, a4) == mapped
    for which in ((0,), (1,), (2,), (3,), (0, 2), (1, 3), (0, 1, 3)):
        st, t, a, arrays = _raw_series(tracks, which, ids, na)
        assert st == S.OK and (t, a) == mapped, which
        for k in which:
            assert arrays[k].tobytes() == full[k].tobytes(), (which, k)


@pytest.mark.gpu
def test_series_do_not_depend_on_entries_chunks_or_devices(monkeypatch):
    import torch

    sr = 44100
    tracks = [R.encode(_multichannel(8, 20 * sr, sr, 41), S.PCM_S16, sr), R.encode(_multichannel(1, 9 * 48000, 48000, 42), S.PCM_F32, 48000),
              R.encode(_multichannel(3, 31 * sr, sr, 43), S.PCM_S24, sr), R.encode(_multichannel(6, 5 * 96000, 96000, 44), S.PCM_U8, 96000),
              R.encode(_multichannel(2, 35 * sr, sr, 45), S.PCM_F64, sr), S.PcmTrack(np.zeros(0, np.uint8), S.PCM_S16, 2, sr)]
    maps = [S.channel_map(0x63F, 8), S.channel_map(0, 1, dual_mono=True), None, S.channel_map(0x60F, 6), None, None]
    ids = [0, 1, 0, None, 1, None]
    kw = dict(channel_maps=maps, series=True)

    def key(ts, als):
        return [(_all([g])[0], _ser(g)) for g in ts], [_full(a) for a in als]

    whole = key(*S.loudness_albums_pcm(tracks, ids, **kw))
    plain_t, plain_a = S.loudness_albums_pcm(tracks, ids, channel_maps=maps)
    assert [x[0] for x in whole[0]] == _all(plain_t) and whole[1] == [_full(a) for a in plain_a]  # the series change no result
    assert key(*S.loudness_albums_pcm(tracks, ids, devices=[0, 0], **kw)) == whole
    _, t, a = S.analyze_loudness_pcm(tracks, albums=ids, **kw)
    assert key(t, a) == whole
    monkeypatch.setenv("STRATUM_B200_STAGE_MB", "1")  # every track in an upload chunk of its own
    assert key(*S.loudness_albums_pcm(tracks, ids, **kw)) == whole
    _, t, a = S.analyze_loudness_pcm(tracks, albums=ids, **kw)
    assert key(t, a) == whole
    monkeypatch.delenv("STRATUM_B200_STAGE_MB")
    cat = np.concatenate([x.data for x in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    d = torch.from_numpy(cat).cuda()
    t, a = S.loudness_albums_pcm_device(d.data_ptr(), offsets, srs, chans, fmts, ids, device=d.device.index, **kw)
    torch.cuda.synchronize()
    assert key(t, a) == whole
    if S.device_count() >= 2:
        assert key(*S.loudness_albums_pcm(tracks, ids, devices=[0, 1], **kw)) == whole


@pytest.mark.gpu
def test_series_across_two_devices():
    if S.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    sr = 48000
    tracks = [R.encode(_multichannel(2 + 2 * i, (10 + 5 * i) * sr, sr, 60 + i), FMTS[i], sr) for i in range(4)]
    one = S.loudness_batch_pcm(tracks, devices=[0], series=True)
    two = S.loudness_batch_pcm(tracks, devices=[0, 1], series=True)
    assert [(_full(g), _ser(g)) for g in two] == [(_full(g), _ser(g)) for g in one]


@pytest.mark.gpu
def test_seven_one_map_weighs_the_loudness_series_but_not_the_peaks():
    sr = 48000
    t = R.encode(_multichannel(8, int(33.5 * sr), sr, 88), S.PCM_S24, sr)
    m = S.channel_map(0x63F, 8)
    mapped, plain = S.loudness_batch_pcm([t, t], channel_maps=[m, None], series=True)
    _check_series(mapped, t, m, "7.1 map")
    _check_series(plain, t, None, "default map")
    assert not np.array_equal(mapped.series.momentary_lufs, plain.series.momentary_lufs)
    assert np.array_equal(mapped.series.sample_peak, plain.series.sample_peak) and np.array_equal(mapped.series.true_peak, plain.series.true_peak)
    _check_maxima(mapped)


def _sine(db, n, sr, f=1000.0):
    x = 10.0 ** (db / 20.0) * np.sin(2 * np.pi * f * np.arange(n) / sr)
    return np.stack([x, x], axis=1)


@pytest.mark.gpu
def test_ebu_tech_3341_signals():
    sr = 48000
    Sb = sr // 10
    level = _sine(-23.0, 20 * sr, sr)
    step = _sine(-33.0, 20 * sr, sr)
    step[10 * sr:] *= 10.0 ** 0.5  # -33 -> -23 dBFS at 10 s, in phase
    click = _sine(-20.0, 12 * sr, sr)
    at = 57 * Sb + 1234
    click[at, 1] = 1.0
    g_level, g_step, g_click = S.loudness_batch_pcm([R.encode(x, S.PCM_F32, sr) for x in (level, step, click)], series=True)
    for k in ("momentary_lufs", "short_term_lufs"):
        v = getattr(g_level.series, k)
        assert v.size > 0 and np.all(np.abs(v - -23.0) <= 0.1), (k, v.min(), v.max())
    m = g_step.series.momentary_lufs
    before, after = m[:100 - 4 + 1], m[100:]  # block j covers segments j .. j + 3; the step starts segment 100
    assert np.all(np.abs(before - -33.0) <= 0.1) and np.all(np.abs(after - -23.0) <= 0.1)
    assert np.all((m[97:100] > -33.0 + 0.1) & (m[97:100] < -23.0 - 0.1))  # the blocks that straddle the step
    sp = g_click.series.sample_peak
    assert sp[at // Sb] == 1.0
    assert np.all(np.delete(sp, at // Sb) < 0.2) and g_click.sample_peak == 1.0
    assert g_click.series.true_peak[at // Sb] >= 1.0


@pytest.mark.gpu
def test_launches_and_read_backs():
    sr = 48000
    tracks = [R.encode(_multichannel(c, int(5.37 * sr), sr, 31 + c), S.PCM_S16, sr) for c in (2, 6, 8)]
    tracks.append(S.PcmTrack(tracks[0].data.copy(), S.PCM_S16, 2, 7999))  # failed: no segments
    n = len(tracks)
    nseg = sum(S.loudness_series_lengths(t.sample_rate, t.frames)[2] for t in tracks)
    assert nseg == 3 * 54
    _raw_series(tracks, (0, 1, 2, 3))  # buffers sized before counting

    def counted(which):
        l0, (_, d0) = S.launch_count(), S.transfer_bytes()
        st, *_ = _raw_series(tracks, which)
        assert st == S.OK
        l1, (_, d1) = S.launch_count(), S.transfer_bytes()
        return l1 - l0, d1 - d0

    assert counted(()) == (4, n * LOUD_OUT_BYTES)
    for which in ((0,), (2,), (1, 3), (0, 1, 2, 3)):
        assert counted(which) == (4, n * LOUD_OUT_BYTES + 8 * nseg * len(which)), which
