"""Analysis and loudness from one upload (stratum_b200_analyze_loudness_pcm): call validation on the CPU; on the GPU, results identical
to stratum_b200_analyze_batch_pcm and stratum_b200_loudness_albums_pcm over a mixed batch, across upload chunks, devices and a
concurrent caller, the PCM counted once in the upload bytes, and the loudness stage times next to the analysis ones."""
import ctypes as C
import dataclasses
import re
import threading
from pathlib import Path

import numpy as np
import pytest

import loudness_ref as R
import stratum_dsp_b200 as S
from test_loudness import _fields, _multichannel, _stereo_c2

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()
U32P, U64P = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_symbol_declared_and_exported():
    assert re.search(r"\bstratum_b200_analyze_loudness_pcm\s*\(", HEADER)
    assert hasattr(S.lib(), "stratum_b200_analyze_loudness_pcm")


def _raw_call(data, offsets, srs, chans, fmts, ids, n_albums, cfg=None, with_out=True, with_loudness_out=True, with_album_out=True):
    n = len(offsets) - 1
    off = np.ascontiguousarray(offsets, np.uint64)
    arr = lambda v: np.ascontiguousarray(v, np.uint32)
    s, c, f = arr(srs), arr(chans), arr(fmts)
    res = (S.StratumResult * max(n, 1))() if with_out else None
    loud = (S.StratumLoudness * max(n, 1))() if with_loudness_out else None
    alb = (S.StratumLoudness * max(n_albums, 1))() if with_album_out else None
    p = lambda a: a.ctypes.data_as(U32P)
    idp = p(arr(ids)) if ids is not None else None
    cfgp = C.cast(C.byref(cfg._c), C.c_void_p) if cfg is not None else None
    st = S.lib().stratum_b200_analyze_loudness_pcm(data.ctypes.data if data is not None else None, off.ctypes.data_as(U64P), p(s), p(c), p(f), n, cfgp,
                                                   idp, n_albums, None, 0, res, loud, alb)
    if res is not None:
        S.lib().stratum_b200_result_free(res, n)
    return st


@pytest.mark.parametrize("case", ["id_out_of_range", "id_with_no_albums", "null_album_of_track", "null_album_out", "unknown_format", "zero_channels",
                                  "too_many_channels", "partial_frame", "null_pcm", "null_out", "null_loudness_out"])
def test_malformed_calls_are_rejected_whole(case):
    data = np.zeros(4 * 100, np.uint8)
    offsets, srs, chans, fmts = [0, 200, 400], [48000, 48000], [2, 2], [S.PCM_S16, S.PCM_S16]
    ids, n_albums, outs = [0, S.NO_ALBUM], 1, {}
    if case == "id_out_of_range":
        ids = [0, 1]
    elif case == "id_with_no_albums":
        ids, n_albums = [S.NO_ALBUM, 0], 0
    elif case == "null_album_of_track":
        ids = None
    elif case == "null_album_out":
        outs = {"with_album_out": False}
    elif case == "unknown_format":
        fmts = [S.PCM_S16, 9]
    elif case == "zero_channels":
        chans = [2, 0]
    elif case == "too_many_channels":
        chans = [2, 65]
    elif case == "partial_frame":
        offsets = [0, 200, 399]
    elif case == "null_pcm":
        data = None
    elif case == "null_out":
        outs = {"with_out": False}
    else:
        outs = {"with_loudness_out": False}
    assert _raw_call(data, offsets, srs, chans, fmts, ids, n_albums, **outs) == S.INVALID_INPUT
    assert S.last_error()


def test_unbuilt_config_switch_is_rejected_before_device_work():
    data = np.zeros(4 * 100, np.uint8)
    st = _raw_call(data, [0, 200, 400], [48000, 48000], [2, 2], [S.PCM_S16, S.PCM_S16], None, 0, cfg=S.AnalysisConfig(frame_size=1024))
    assert st == S.NOT_IMPLEMENTED
    assert "frame_size" in S.last_error()


def test_config_is_checked_before_the_pcm_layout_as_in_the_analysis_entry():
    data = np.zeros(4 * 100, np.uint8)
    st = _raw_call(data, [0, 200, 399], [48000, 48000], [2, 2], [S.PCM_S16, S.PCM_S16], None, 0, cfg=S.AnalysisConfig(frame_size=1024))
    assert st == S.NOT_IMPLEMENTED
    res = (S.StratumResult * 2)()
    p = lambda v: np.ascontiguousarray(v, np.uint32).ctypes.data_as(U32P)
    off = np.array([0, 200, 399], np.uint64)
    cfg = S.AnalysisConfig(frame_size=1024)
    assert S.lib().stratum_b200_analyze_batch_pcm(C.c_void_p(data.ctypes.data), off.ctypes.data_as(U64P), p([48000, 48000]), p([2, 2]),
                                                  p([S.PCM_S16, S.PCM_S16]), C.c_uint32(2), C.cast(C.byref(cfg._c), C.c_void_p), None, C.c_uint32(0),
                                                  res) == st


def test_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    t = R.encode(np.zeros((48000, 2)), S.PCM_S16, 48000)
    with pytest.raises(S.AnalysisError) as e:
        S.analyze_loudness_pcm([t], albums=[0])
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message


def test_python_album_ids_are_checked():
    t = R.encode(np.zeros((4800, 2)), S.PCM_S16, 48000)
    with pytest.raises(ValueError):
        S.analyze_loudness_pcm([t, t], albums=[0])
    with pytest.raises(ValueError):
        S.analyze_loudness_pcm([t], albums=[-1])
    with pytest.raises(ValueError):
        S.analyze_loudness_pcm([t], n_albums=2)


# ---- GPU -----------------------------------------------------------------------------------------------------------------
_ARRAYS = {"beats": "n_beats", "downbeats": "n_downbeats", "bars": "n_bars", "onsets": "n_onsets", "hmm_beat_frames": "n_hmm_beat_frames",
           "tempogram_candidates": "n_tempogram_candidates"}


def _raw(r, skip=()) -> tuple:
    """Every field of a result struct but those in skip, as bytes (padding excluded); the arrays of a StratumResult by content."""
    out = []
    for name, ty in type(r)._fields_:
        if name in skip:
            continue
        if name == "error":
            out.append(r.error)
        elif name in _ARRAYS:
            n = max(getattr(r, _ARRAYS[name]), 0)
            out.append(C.string_at(getattr(r, name), n * C.sizeof(ty._type_)) if n else b"")
        else:
            out.append(C.string_at(C.addressof(r) + getattr(type(r), name).offset, C.sizeof(ty)))
    return tuple(out)


def _raw_result(r: S.StratumResult) -> tuple:
    return _raw(r, skip=("processing_time_ms",))


_loud_raw = _raw


def _py(v):
    """A Python-surface result as plain comparable values: floats by their bits, arrays by dtype and bytes."""
    if dataclasses.is_dataclass(v):
        return tuple(_py(getattr(v, f.name)) for f in dataclasses.fields(v))
    if isinstance(v, np.ndarray):
        return v.dtype.str, v.tobytes()
    if isinstance(v, float):
        return v.hex()
    if isinstance(v, (list, tuple)):
        return tuple(_py(x) for x in v)
    if isinstance(v, S.AnalysisError):
        return v.code, v.message
    return v


def _tables(tracks):
    cat = np.concatenate([t.data for t in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    return cat, offsets, srs, chans, fmts


def _analyze_batch_pcm(tracks, res, dev=None, nd=0):
    """stratum_b200_analyze_batch_pcm into res (every argument typed here: the library declares this entry's types lazily)."""
    cat, offsets, srs, chans, fmts = _tables(tracks)
    st = S.lib().stratum_b200_analyze_batch_pcm(C.c_void_p(cat.ctypes.data), offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P),
                                                chans.ctypes.data_as(U32P), fmts.ctypes.data_as(U32P), C.c_uint32(len(tracks)), None, dev,
                                                C.c_uint32(nd), res)
    assert st == S.OK, S.last_error()


def _separate(tracks, ids, n_albums, devices=None):
    """stratum_b200_analyze_batch_pcm, then stratum_b200_loudness_albums_pcm."""
    n = len(tracks)
    cat, offsets, srs, chans, fmts = _tables(tracks)
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    nd = len(devices) if devices else 0
    res = (S.StratumResult * n)()
    loud, alb = (S.StratumLoudness * n)(), (S.StratumLoudness * max(n_albums, 1))()
    L = S.lib()
    _analyze_batch_pcm(tracks, res, dev, nd)
    st = L.stratum_b200_loudness_albums_pcm(cat.ctypes.data, offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P), chans.ctypes.data_as(U32P),
                                            fmts.ctypes.data_as(U32P), n, ids.ctypes.data_as(U32P), n_albums, dev, nd, loud, alb)
    assert st == S.OK, S.last_error()
    try:
        return [_raw_result(r) for r in res], [_loud_raw(r) for r in loud], [_loud_raw(a) for a in alb[:n_albums]]
    finally:
        L.stratum_b200_result_free(res, n)


def _combined(tracks, ids, n_albums, devices=None):
    n = len(tracks)
    cat, offsets, srs, chans, fmts = _tables(tracks)
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    res = (S.StratumResult * n)()
    loud, alb = (S.StratumLoudness * n)(), (S.StratumLoudness * max(n_albums, 1))()
    L = S.lib()
    st = L.stratum_b200_analyze_loudness_pcm(cat.ctypes.data, offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P), chans.ctypes.data_as(U32P),
                                             fmts.ctypes.data_as(U32P), n, None, ids.ctypes.data_as(U32P), n_albums, dev, len(devices) if devices else 0,
                                             res, loud, alb)
    assert st == S.OK, S.last_error()
    try:
        return [_raw_result(r) for r in res], [_loud_raw(r) for r in loud], [_loud_raw(a) for a in alb[:n_albums]]
    finally:
        L.stratum_b200_result_free(res, n)


_BATCH = None


def _mixed_batch():
    """Six formats, 1 / 2 / 6 channels, 44.1 / 48 / 96 kHz, 0.3 s to 3 min, an all-zero track, a 0-frame track and a track at 7999 Hz;
    album 0 is measured, album 1 has the 0-frame member, album 2 is named by no track."""
    global _BATCH
    if _BATCH is None:
        tracks = [R.encode(_stereo_c2(0, 7_938_000, 44100), S.PCM_S16, 44100),
                  R.encode(_multichannel(6, 20 * 48000, 48000, 1), S.PCM_F32, 48000),
                  R.encode(_multichannel(1, int(0.3 * 96000), 96000, 2), S.PCM_S24, 96000),
                  R.encode(np.zeros((10 * 48000, 2)), S.PCM_S16, 48000),
                  S.PcmTrack(np.zeros(0, np.uint8), S.PCM_U8, 2, 44100),
                  S.PcmTrack(R.encode(_multichannel(1, 12 * 8000, 8000, 3), S.PCM_S32, 8000).data, S.PCM_S32, 1, 7999),
                  R.encode(_stereo_c2(6, 30 * 44100, 44100), S.PCM_F64, 44100),
                  R.encode(_multichannel(2, 15 * 96000, 96000, 4), S.PCM_U8, 96000)]
        ids = np.array([0, 0, 1, S.NO_ALBUM, 1, S.NO_ALBUM, 0, 1], np.uint32)
        _BATCH = tracks, ids, 3
    return _BATCH


@pytest.mark.gpu
def test_results_equal_the_two_separate_entries():
    tracks, ids, na = _mixed_batch()
    ana, loud, alb = _combined(tracks, ids, na)
    assert (ana, loud, alb) == _separate(tracks, ids, na)
    # the batch covers what it claims: independent per-track failures and album failures
    results, per_track, albums = S.analyze_loudness_pcm(tracks, albums=[None if i == S.NO_ALBUM else int(i) for i in ids], n_albums=na)
    assert results[3].error is not None and "silent" in results[3].error.message and per_track[3].error is None
    assert per_track[5].error.kind == "NotImplemented" and per_track[4].error.kind == "InvalidInput"
    assert results[0].error is None and per_track[0].error is None and results[0].bpm > 0
    assert albums[0].error is None and albums[1].error.message.startswith("track 4:") and albums[2].error.message == "album has no tracks"
    # the Python surface returns what the two Python entries return
    sep_res = S.analyze_batch_pcm(tracks)
    sep_loud, sep_alb = S.loudness_albums_pcm(tracks, [None if i == S.NO_ALBUM else int(i) for i in ids], n_albums=na)
    for a, b in zip(results, sep_res):
        a.metadata.processing_time_ms = b.metadata.processing_time_ms = 0.0
    assert [_py(a) for a in results] == [_py(b) for b in sep_res]
    assert [_fields(g) for g in per_track] == [_fields(g) for g in sep_loud]
    assert [_fields(g) for g in albums] == [_fields(g) for g in sep_alb]
    assert S.analyze_loudness_pcm(tracks[:2])[2] == []


@pytest.mark.gpu
def test_results_equal_the_two_separate_entries_across_upload_chunks(monkeypatch):
    tracks, ids, na = _mixed_batch()
    whole = _combined(tracks, ids, na)
    # chunks of 1 MB of mono f32 frames: every track lands in a chunk of its own, and the batch spans several staging rounds
    monkeypatch.setenv("STRATUM_B200_STAGE_MB", "1")
    split = _combined(tracks, ids, na)
    assert split == _separate(tracks, ids, na)
    assert split == whole


@pytest.mark.gpu
def test_the_pcm_is_uploaded_once():
    sr = 44100
    tracks = [R.encode(_stereo_c2(10 + i, 40 * sr, sr), S.PCM_S16, sr) for i in range(3)]
    ids = np.array([0, 0, 1], np.uint32)
    _separate(tracks, ids, 2)  # per-sample-rate tables and buffers built before counting

    def counters():
        h2d, d2h = S.transfer_bytes()
        return S.launch_count(), h2d, d2h

    c0 = counters()
    _separate(tracks, ids, 2)
    c1 = counters()
    _combined(tracks, ids, 2)
    c2 = counters()
    sep = [b - a for a, b in zip(c0, c1)]
    comb = [b - a for a, b in zip(c1, c2)]
    pcm = sum(t.data.size for t in tracks)
    assert comb[0] == sep[0]  # launches
    assert comb[2] == sep[2]  # device to host
    assert comb[1] == sep[1] - pcm  # host to device: the PCM once instead of twice


@pytest.mark.gpu
def test_stage_times_show_both_halves():
    sr = 48000
    tracks = [R.encode(_multichannel(2, 20 * sr, sr, 70 + i), S.PCM_S16, sr) for i in range(2)]
    S.stage_timing(True)
    try:
        S.stage_times(reset=True)
        S.analyze_loudness_pcm(tracks, albums=[0, 0])
        names = set(S.stage_times(reset=True))
    finally:
        S.stage_timing(False)
    for s in ("loudness_pass1", "loudness_scan", "loudness_pass2", "loudness_gate", "loudness_album_gate", "final_bpm", "beats"):
        assert s in names, (s, sorted(names))


@pytest.mark.gpu
def test_devices():
    tracks, ids, na = _mixed_batch()
    one = _combined(tracks, ids, na)
    assert _combined(tracks, ids, na, devices=[0, 0]) == one
    if S.device_count() < 2:
        pytest.skip("the two-device case needs two CUDA devices")
    assert _combined(tracks, ids, na, devices=[0, 1]) == one


@pytest.mark.gpu
def test_concurrent_callers_on_one_device():
    tracks, ids, na = _mixed_batch()
    other = [R.encode(_multichannel(2, 25 * 44100, 44100, 80 + i), S.PCM_S24, 44100) for i in range(3)]

    def analyze_other():
        res = (S.StratumResult * len(other))()
        _analyze_batch_pcm(other, res)
        try:
            return [_raw_result(r) for r in res]
        finally:
            S.lib().stratum_b200_result_free(res, len(other))

    serial = (_combined(tracks, ids, na), analyze_other())
    got = [None, None]

    def run(k):
        got[k] = _combined(tracks, ids, na) if k == 0 else analyze_other()

    th = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert tuple(got) == serial
