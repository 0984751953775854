"""Album loudness (stratum_b200_loudness_albums_pcm): call validation on the CPU; on the GPU, per-track results identical to the
batch entry, an album of one track identical to the track, parity with the float64 album rule of loudness_album_ref.py, pooling rather
than averaging, bit-identical album values across layouts, chunks, entries and devices, and album failures."""
import ctypes as C
import math
import re
from pathlib import Path

import numpy as np
import pytest

import loudness_album_ref as RA
import loudness_ref as R
import stratum_dsp_b200 as S
import synth
from test_loudness import FIELDS, _fields, _multichannel, _sine, _stereo_c2

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()
FMTS = [S.PCM_U8, S.PCM_S16, S.PCM_S24, S.PCM_S32, S.PCM_F32, S.PCM_F64]


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_album_symbols_declared_and_exported():
    L = S.lib()
    for s in ("stratum_b200_loudness_albums_pcm", "stratum_b200_loudness_albums_pcm_device"):
        assert re.search(rf"\b{s}\s*\(", HEADER), s
        assert hasattr(L, s), s
    m = re.search(r"#define STRATUM_NO_ALBUM (0x[0-9A-Fa-f]+)u", HEADER)
    assert m and int(m.group(1), 16) == S.NO_ALBUM == 0xFFFFFFFF


def _raw_album_call(device_entry, data, offsets, srs, chans, fmts, ids, n_albums, with_album_out=True):
    n = len(offsets) - 1
    off = np.ascontiguousarray(offsets, np.uint64)
    arr = lambda v: np.ascontiguousarray(v, np.uint32)
    s, c, f = arr(srs), arr(chans), arr(fmts)
    res = (S.StratumLoudness * max(n, 1))()
    alb = (S.StratumLoudness * max(n_albums, 1))() if with_album_out else None
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint32))
    idp = p(arr(ids)) if ids is not None else None
    if device_entry:  # the address is never dereferenced: every case stops in the validation
        pcm = C.c_void_p(1 << 20) if data is not None else None
        return S.lib().stratum_b200_loudness_albums_pcm_device(pcm, off.ctypes.data_as(C.POINTER(C.c_uint64)), p(s), p(c), p(f), n, idp, n_albums, 0,
                                                               res, alb)
    return S.lib().stratum_b200_loudness_albums_pcm(data.ctypes.data if data is not None else None, off.ctypes.data_as(C.POINTER(C.c_uint64)), p(s),
                                                    p(c), p(f), n, idp, n_albums, None, 0, res, alb)


@pytest.mark.parametrize("device_entry", [False, True])
@pytest.mark.parametrize("case", ["id_out_of_range", "id_with_no_albums", "null_album_of_track", "null_album_out", "unknown_format", "zero_channels",
                                  "too_many_channels", "partial_frame", "null_pcm"])
def test_malformed_album_calls_are_rejected_whole(case, device_entry):
    data = np.zeros(4 * 100, np.uint8)
    offsets, srs, chans, fmts = [0, 200, 400], [48000, 48000], [2, 2], [S.PCM_S16, S.PCM_S16]
    ids, n_albums, with_album_out = [0, S.NO_ALBUM], 1, True
    if case == "id_out_of_range":
        ids = [0, 1]
    elif case == "id_with_no_albums":
        ids, n_albums = [S.NO_ALBUM, 0], 0
    elif case == "null_album_of_track":
        ids = None
    elif case == "null_album_out":
        with_album_out = False
    elif case == "unknown_format":
        fmts = [S.PCM_S16, 9]
    elif case == "zero_channels":
        chans = [2, 0]
    elif case == "too_many_channels":
        chans = [2, 65]
    elif case == "partial_frame":
        offsets = [0, 200, 399]
    else:
        data = None
    assert _raw_album_call(device_entry, data, offsets, srs, chans, fmts, ids, n_albums, with_album_out) == S.INVALID_INPUT
    assert S.last_error()


def test_python_album_ids_are_checked():
    t = R.encode(np.zeros((4800, 2)), S.PCM_S16, 48000)
    with pytest.raises(ValueError):
        S.loudness_albums_pcm([t, t], [0])
    with pytest.raises(ValueError):
        S.loudness_albums_pcm([t], [-1])


@pytest.mark.parametrize("sr,C,seconds,fmt", [(44100, 2, 12.0, S.PCM_S16), (48000, 6, 2.5, S.PCM_F32), (96000, 1, 0.3, S.PCM_S24)])
def test_album_reference_of_one_track_is_the_track_reference(sr, C, seconds, fmt):
    t = R.encode(_multichannel(C, int(seconds * sr), sr, 7), fmt, sr)
    album, track = RA.measure_album([t]), R.measure(t)
    assert album.pop("frames") == t.frames
    assert album == track


def test_album_entries_have_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    t = R.encode(np.zeros((48000, 2)), S.PCM_S16, 48000)
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_albums_pcm([t], [0])
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_albums_pcm_device(1 << 20, np.array([0, t.data.size], np.uint64), [48000], [2], [S.PCM_S16], [0])
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message


# ---- GPU -----------------------------------------------------------------------------------------------------------------
def _full(g: S.Loudness):
    return _fields(g) + ((g.error.kind, g.error.message) if g.error else (None, None),)


def _check_album(g: S.Loudness, ref: dict, label=""):
    assert g.error is None, f"{label}: {g.error}"
    assert (g.n_momentary, g.n_short_term, g.frames) == (ref["n_momentary"], ref["n_short_term"], ref["frames"]), label
    assert g.sample_rate == 0 and g.channels == 0, label
    for f, tol in (("integrated_lufs", 0.01), ("momentary_max_lufs", 0.01), ("short_term_max_lufs", 0.01), ("loudness_range_lu", 0.02)):
        a, b = getattr(g, f), ref[f]
        if math.isinf(b):
            assert a == b, f"{label} {f}: {a} vs {b}"
        else:
            assert abs(a - b) <= tol, f"{label} {f}: {a} vs {b}"
    assert g.sample_peak == ref["sample_peak"], label
    assert abs(g.true_peak - ref["true_peak"]) <= 1e-5 * ref["true_peak"], f"{label} true_peak: {g.true_peak} vs {ref['true_peak']}"


def _mixed_batch(sr):
    """The batch of test_loudness.py::test_parity_formats_channels_lengths."""
    Sb = (sr + 5) // 10
    lengths = [int(0.3 * sr), 4 * Sb, int(2.9 * sr), 30 * Sb, 20 * sr]
    chans = [1, 2, 6, 8, 5, 4]
    tracks = []
    for i, n in enumerate(lengths):
        for j in range(2):
            q = (i * 2 + j) % len(FMTS)
            tracks.append(R.encode(_multichannel(chans[(i + 3 * j) % len(chans)], n, sr, 100 * i + j), FMTS[q], sr))
    return tracks


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [44100, 48000])
def test_per_track_results_equal_the_batch_entry(sr):
    tracks = _mixed_batch(sr)
    ids = [None if i % 4 == 3 else i % 3 for i in range(len(tracks))]
    got, albums = S.loudness_albums_pcm(tracks, ids)
    assert len(albums) == 3 and all(a.error is None for a in albums)
    assert [_full(g) for g in got] == [_full(g) for g in S.loudness_batch_pcm(tracks)]


@pytest.mark.gpu
def test_album_of_one_track_is_that_track():
    sr = 44100
    tracks = [R.encode(_stereo_c2(5, 7_938_000, sr), S.PCM_S16, sr),  # three minutes
              R.encode(_multichannel(2, int(2.5 * sr), sr, 11), S.PCM_S24, sr),  # K = 0
              R.encode(_multichannel(2, int(0.3 * sr), sr, 12), S.PCM_F32, sr)]  # J = 0
    got, albums = S.loudness_albums_pcm(tracks, [0, 1, 2])
    assert albums[1].n_short_term == 0 and albums[2].n_momentary == 0
    keep = [f for f in FIELDS if f not in ("sample_rate", "channels")]
    for t, a in zip(got, albums):
        assert a.error is None and t.error is None
        assert [getattr(a, f) for f in keep] == [getattr(t, f) for f in keep]
        assert a.sample_rate == 0 and a.channels == 0


@pytest.mark.gpu
def test_parity_mixed_rates_channels_formats():
    specs = [(44100, 1, 12.0), (48000, 2, 25.0), (96000, 6, 8.0), (44100, 8, 31.0), (48000, 5, 4.5), (96000, 4, 17.0), (44100, 2, 40.0),
             (48000, 1, 2.0), (96000, 3, 9.0)]
    tracks = [R.encode(_multichannel(c, int(d * sr), sr, 40 + i), FMTS[i % len(FMTS)], sr) for i, (sr, c, d) in enumerate(specs)]
    ids = [i % 3 for i in range(len(tracks))]  # every album mixes the three rates
    _, albums = S.loudness_albums_pcm(tracks, ids)
    for a in range(3):
        _check_album(albums[a], RA.measure_album([t for t, i in zip(tracks, ids) if i == a]), f"album {a}")


@pytest.mark.gpu
def test_parity_album_with_the_sixty_minute_mix():
    sr = 44100
    c4 = R.encode(synth.c4_mix(), S.PCM_F32, sr)
    tracks = [R.encode(_stereo_c2(9, 60 * sr, sr), S.PCM_S16, sr), c4, R.encode(_multichannel(6, 20 * 48000, 48000, 77), S.PCM_S24, 48000)]
    _, (album,) = S.loudness_albums_pcm(tracks, [0, 0, 0])
    _check_album(album, RA.measure_album(tracks), "c4 album")


def _sine_track(db, seconds=20.0):
    return R.encode(_sine(db, seconds), S.PCM_F32, 48000)


@pytest.mark.gpu
def test_album_range_pools_the_short_term_values():
    tracks = [_sine_track(-20.0), _sine_track(-30.0)]
    got, (album,) = S.loudness_albums_pcm(tracks, [0, 0])
    assert abs(album.loudness_range_lu - 10.0) <= 0.1, album
    assert all(abs(g.loudness_range_lu) <= 0.1 for g in got), got


@pytest.mark.gpu
def test_quiet_track_falls_under_the_album_gate():
    loud, quiet = _sine_track(-23.0), _sine_track(-38.0)
    got, (album,) = S.loudness_albums_pcm([loud, quiet], [0, 0])
    li, qi = got[0].integrated_lufs, got[1].integrated_lufs
    assert abs(li + 23.0) <= 0.1 and abs(qi + 38.0) <= 0.1, got
    assert abs(album.integrated_lufs - li) <= 0.05, album
    power_mean = -0.691 + 10 * math.log10((10 ** ((li + 0.691) / 10) + 10 ** ((qi + 0.691) / 10)) / 2)
    assert album.integrated_lufs - power_mean > 2.0, (album.integrated_lufs, power_mean)


@pytest.mark.gpu
def test_near_silent_track_leaves_the_album_unchanged():
    a, b, silent = _sine_track(-20.0), _sine_track(-26.0), _sine_track(-80.0)
    _, (two,) = S.loudness_albums_pcm([a, b], [0, 0])
    _, (three,) = S.loudness_albums_pcm([a, b, silent], [0, 0, 0])
    assert abs(three.integrated_lufs - two.integrated_lufs) <= 0.01, (two, three)


@pytest.mark.gpu
def test_album_values_do_not_depend_on_layout_chunks_entry_or_devices(monkeypatch):
    import torch

    sr = 44100
    members = [R.encode(_stereo_c2(3, 30 * sr, sr), S.PCM_S16, sr), R.encode(_multichannel(6, 12 * 48000, 48000, 21), S.PCM_F32, 48000),
               R.encode(_multichannel(1, 35 * sr, sr, 22), S.PCM_S24, sr)]
    others = [R.encode(_multichannel(2, 3 * 96000, 96000, 23), S.PCM_S16, 96000), R.encode(_multichannel(8, 40 * sr, sr, 24), S.PCM_U8, sr),
              R.encode(_multichannel(4, 9 * sr, sr, 25), S.PCM_F64, sr)]
    _, (alone,) = S.loudness_albums_pcm(members, [0, 0, 0])
    alone = _full(alone)
    batch = [others[0], members[0], others[1], members[1], others[2], members[2]]
    ids = [1, 0, None, 0, 1, 0]
    _, albums = S.loudness_albums_pcm(batch, ids)
    assert _full(albums[0]) == alone
    _, albums = S.loudness_albums_pcm(batch, ids, devices=[0, 0])
    assert _full(albums[0]) == alone
    whole = [_full(a) for a in albums]
    # chunks of 1 MB of mono f32 frames: every track lands in a chunk of its own
    monkeypatch.setenv("STRATUM_B200_STAGE_MB", "1")
    _, split = S.loudness_albums_pcm(batch, ids)
    monkeypatch.delenv("STRATUM_B200_STAGE_MB")
    assert [_full(a) for a in split] == whole
    cat = np.concatenate([t.data for t in batch])
    offsets = np.zeros(len(batch) + 1, np.uint64)
    offsets[1:] = np.cumsum([t.data.size for t in batch])
    d = torch.from_numpy(cat).cuda()
    _, dev = S.loudness_albums_pcm_device(d.data_ptr(), offsets, [t.sample_rate for t in batch], [t.channels for t in batch], [t.fmt for t in batch],
                                          ids, device=d.device.index)
    torch.cuda.synchronize()
    assert [_full(a) for a in dev] == whole


@pytest.mark.gpu
def test_album_launches():
    sr = 48000
    tracks = [R.encode(_multichannel(2, 5 * sr, sr, 31 + i), S.PCM_S16, sr) for i in range(3)]
    n0 = S.launch_count()
    S.loudness_batch_pcm(tracks)
    n1 = S.launch_count()
    S.loudness_albums_pcm(tracks, [None, None, None])
    n2 = S.launch_count()
    S.loudness_albums_pcm(tracks, [0, 0, 1])
    n3 = S.launch_count()
    assert n1 - n0 == 4  # one chunk: pass 1, scan, pass 2, gate
    assert n2 - n1 == 4
    assert n3 - n2 == 5


@pytest.mark.gpu
def test_failing_albums_fail_alone():
    sr = 48000
    good = [R.encode(_multichannel(2, (5 + i) * sr, sr, 50 + i), S.PCM_S16, sr) for i in range(4)]
    empty = S.PcmTrack(np.zeros(0, np.uint8), S.PCM_S16, 2, sr)
    low = S.PcmTrack(good[3].data.copy(), S.PCM_S16, 2, 7999)
    batch = [good[0], good[1], empty, good[2], good[3], low, empty]
    ids = [0, 0, 1, 1, 2, 2, 2]  # album 3 is named by no track
    got, albums = S.loudness_albums_pcm(batch, ids, n_albums=4)
    ref_tracks, (ref_album,) = S.loudness_albums_pcm(good[:2], [0, 0])
    assert _full(albums[0]) == _full(ref_album)
    assert [_full(got[i]) for i in (0, 1)] == [_full(g) for g in ref_tracks]
    singles = S.loudness_batch_pcm([good[2], good[3]])
    assert _full(got[3]) == _full(singles[0]) and _full(got[4]) == _full(singles[1])
    a1, a2, a3 = albums[1], albums[2], albums[3]
    assert a1.error.kind == "InvalidInput" and a1.error.message.startswith("track 2: empty track"), a1.error
    assert a2.error.kind == "NotImplemented" and a2.error.message.startswith("track 5: sample rate 7999 Hz"), a2.error  # the lowest failed member
    assert a3.error.kind == "InvalidInput" and a3.error.message == "album has no tracks", a3.error
    for a in (a1, a2, a3):
        assert a.frames == 0 and a.n_momentary == 0 and a.sample_peak == 0.0


@pytest.mark.gpu
def test_album_across_two_devices():
    if S.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    sr = 44100
    tracks = [R.encode(_multichannel(2, (20 + 5 * i) * sr, sr, 60 + i), FMTS[i], sr) for i in range(4)]
    one_t, one_a = S.loudness_albums_pcm(tracks, [0, 0, 0, 0], devices=[0])
    two_t, two_a = S.loudness_albums_pcm(tracks, [0, 0, 0, 0], devices=[0, 1])
    assert [_full(a) for a in two_a] == [_full(a) for a in one_a]
    assert [_full(g) for g in two_t] == [_full(g) for g in one_t]
