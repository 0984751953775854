"""Channel maps, dual mono and per-channel results of the loudness measurement (stratum_b200_loudness_mapped_pcm and its device and
combined forms, stratum_b200_loudness_channel_map): the mask -> class rule and call validation on the CPU; on the GPU, default-class
maps identical to no map, mapped layouts against the float64 reference of loudness_layout_ref.py, per-channel results identical to
one-channel tracks, mapped albums, invariance across chunks, entries and devices, and the launches and read-backs."""
import ctypes as C
import math
import re
import struct
from pathlib import Path

import numpy as np
import pytest

import loudness_layout_ref as RL
import loudness_ref as R
import stratum_dsp_b200 as S
from test_analyze_loudness import _py
from test_loudness import FIELDS, _fields, _multichannel, _stereo_c2

ROOT = Path(__file__).resolve().parent.parent
HEADER = (ROOT / "include" / "stratum_b200.h").read_text()
FMTS = [S.PCM_U8, S.PCM_S16, S.PCM_S24, S.PCM_S32, S.PCM_F32, S.PCM_F64]
U8P, U32P, U64P = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)
F, SU, U, D = S.CH_FRONT, S.CH_SURROUND, S.CH_UNUSED, S.CH_DUAL_MONO
LOUD_OUT_BYTES = 40  # csrc/kernels.h: LoudOut, the device-to-host record of one result


# ---- CPU -----------------------------------------------------------------------------------------------------------------
def test_symbols_and_classes_declared_and_exported():
    L = S.lib()
    for s in ("stratum_b200_loudness_mapped_pcm", "stratum_b200_loudness_mapped_pcm_device", "stratum_b200_analyze_loudness_mapped_pcm",
              "stratum_b200_loudness_channel_map"):
        assert re.search(rf"\b{s}\s*\(", HEADER), s
        assert hasattr(L, s), s
    for name, v in (("UNUSED", U), ("FRONT", F), ("SURROUND", SU), ("DUAL_MONO", D)):
        assert re.search(rf"\bSTRATUM_CH_{name} = {v}\b", HEADER), name


# (mask, classes without dual mono); dual mono changes only a one-channel track whose class is not UNUSED
MASKS = [(0x4, [F]), (0x3, [F, F]), (0xB, [F, F, U]), (0x33, [F, F, SU, SU]), (0x107, [F, F, F, F]), (0x37, [F, F, F, SU, SU]),
         (0x3F, [F, F, F, U, SU, SU]), (0x60F, [F, F, F, U, SU, SU]), (0x63F, [F, F, F, U, F, F, SU, SU])]


@pytest.mark.parametrize("dual_mono", [False, True])
@pytest.mark.parametrize("mask,classes", MASKS)
def test_channel_map_of_wave_masks(mask, classes, dual_mono):
    want = list(classes)
    if dual_mono and len(want) == 1:
        want = [D]
    assert S.channel_map(mask, len(classes), dual_mono=dual_mono) == want


@pytest.mark.parametrize("C_", range(1, 9))
def test_mask_zero_is_the_default_map(C_):
    by_weight = {0.0: U, 1.0: F, 1.41: SU}
    assert S.channel_map(0, C_) == [by_weight[w] for w in R.weights(C_)]
    assert S.channel_map(0, C_, dual_mono=True) == ([D] if C_ == 1 else [by_weight[w] for w in R.weights(C_)])


def test_channels_beyond_the_mask_are_unused():
    assert S.channel_map(0x3, 4) == [F, F, U, U]
    assert S.channel_map(0x8, 1, dual_mono=True) == [U]  # an LFE-only track stays unused
    assert S.channel_map(0x40000 | 0x3, 3) == [F, F, U]  # reserved bits name no loudspeaker


def test_channel_map_of_a_track_reads_its_mask():
    t = S.PcmTrack(np.zeros(6 * 2 * 10, np.uint8), S.PCM_S16, 6, 48000, 0x60F)
    assert S.channel_map(t) == [F, F, F, U, SU, SU]
    assert S.channel_map(S.PcmTrack(t.data, S.PCM_S16, 6, 48000)) == S.channel_map(0, 6)


@pytest.mark.parametrize("channels", [0, 65])
def test_channel_map_rejects_bad_channel_counts(channels):
    buf = np.zeros(70, np.uint8)
    assert S.lib().stratum_b200_loudness_channel_map(0x3, channels, 0, buf.ctypes.data_as(U8P)) == S.INVALID_INPUT
    assert S.lib().stratum_b200_loudness_channel_map(0x3, 2, 0, None) == S.INVALID_INPUT


def _wav_extensible(path, pcm16: np.ndarray, sr: int, mask: int):
    ch = pcm16.shape[1]
    data = pcm16.astype("<i2").tobytes()
    guid = struct.pack("<H", 1) + bytes.fromhex("000000001000800000aa00389b71")
    fmt = struct.pack("<HHIIHHHHI", 0xFFFE, ch, sr, sr * 2 * ch, 2 * ch, 16, 22, 16, mask) + guid
    body = b"WAVE" + b"fmt " + struct.pack("<I", len(fmt)) + fmt + b"data" + struct.pack("<I", len(data)) + data
    Path(path).write_bytes(b"RIFF" + struct.pack("<I", len(body)) + body)


def test_read_wav_keeps_the_extensible_channel_mask(tmp_path):
    x = (np.arange(8 * 100).reshape(100, 8) % 200 - 100).astype(np.int16)
    _wav_extensible(tmp_path / "a.wav", x, 48000, 0x63F)
    t = S.read_wav(tmp_path / "a.wav")
    assert (t.channels, t.fmt, t.sample_rate, t.channel_mask) == (8, S.PCM_S16, 48000, 0x63F)
    assert np.array_equal(t.data.view("<i2").reshape(-1, 8), x)
    assert S.channel_map(t) == [F, F, F, U, F, F, SU, SU]
    plain = R.encode(np.zeros((10, 2)), S.PCM_S16, 48000)
    assert plain.channel_mask == 0


def _raw_mapped(entry, data, offsets, srs, chans, fmts, ids, n_albums, cmap, cfg=None, with_channel_out=True):
    n = len(offsets) - 1
    off = np.ascontiguousarray(offsets, np.uint64)
    arr = lambda v: np.ascontiguousarray(v, np.uint32)
    s, c, f = arr(srs), arr(chans), arr(fmts)
    p = lambda a: a.ctypes.data_as(U32P)
    idp = p(arr(ids)) if ids is not None else None
    m = np.ascontiguousarray(cmap, np.uint8) if cmap is not None else None
    mp = m.ctypes.data_as(U8P) if m is not None else None
    res = (S.StratumLoudness * max(n, 1))()
    alb = (S.StratumLoudness * max(n_albums, 1))()
    chout = (S.StratumLoudness * max(int(sum(chans)), 1))() if with_channel_out else None
    L = S.lib()
    if entry == "device":  # the address is never dereferenced: every case stops in the validation
        return L.stratum_b200_loudness_mapped_pcm_device(C.c_void_p(1 << 20) if data is not None else None, off.ctypes.data_as(U64P), p(s), p(c), p(f), n,
                                                         idp, n_albums, mp, 0, res, alb, chout)
    pcm = data.ctypes.data if data is not None else None
    if entry == "host":
        return L.stratum_b200_loudness_mapped_pcm(pcm, off.ctypes.data_as(U64P), p(s), p(c), p(f), n, idp, n_albums, mp, None, 0, res, alb, chout)
    out = (S.StratumResult * max(n, 1))()
    cfgp = C.cast(C.byref(cfg._c), C.c_void_p) if cfg is not None else None
    st = L.stratum_b200_analyze_loudness_mapped_pcm(pcm, off.ctypes.data_as(U64P), p(s), p(c), p(f), n, cfgp, idp, n_albums, mp, None, 0, out, res, alb,
                                                    chout)
    L.stratum_b200_result_free(out, n)
    return st


@pytest.mark.parametrize("entry", ["host", "device", "combined"])
@pytest.mark.parametrize("case", ["bad_code", "bad_code_second_track", "partial_frame_first", "album_id_first", "null_out_first", "config_first"])
def test_bad_class_codes_are_rejected_after_every_other_check(entry, case):
    data = np.zeros(4 * 100, np.uint8)
    offsets, srs, chans, fmts = [0, 200, 400], [48000, 48000], [2, 1], [S.PCM_S16, S.PCM_S32]
    ids, n_albums, cfg = [0, S.NO_ALBUM], 1, None
    cmap = [F, 4, F]
    if case == "bad_code_second_track":
        cmap = [F, F, 255]
    elif case == "partial_frame_first":
        offsets = [0, 200, 399]
    elif case == "album_id_first":
        ids = [0, 1]
    elif case == "null_out_first":
        data = None
    elif case == "config_first":
        if entry != "combined":
            pytest.skip("only the combined entry takes a configuration")
        cfg = S.AnalysisConfig(frame_size=1024)
    st = _raw_mapped(entry, data, offsets, srs, chans, fmts, ids, n_albums, cmap, cfg)
    msg = S.last_error()
    if case == "config_first":
        assert st == S.NOT_IMPLEMENTED and "frame_size" in msg
        return
    assert st == S.INVALID_INPUT
    if case.startswith("bad_code"):
        where = "track 1 channel 0" if case == "bad_code_second_track" else "track 0 channel 1"
        assert f"{where}: channel class" in msg, msg
    else:
        assert "channel class" not in msg, msg


def test_python_channel_maps_are_checked():
    t = R.encode(np.zeros((4800, 2)), S.PCM_S16, 48000)
    with pytest.raises(ValueError):
        S.loudness_batch_pcm([t, t], channel_maps=[[F, F]])
    with pytest.raises(ValueError):
        S.loudness_batch_pcm([t], channel_maps=[[F, F, F]])
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_batch_pcm([t], channel_maps=[[F, 7]])
    assert e.value.kind == "InvalidInput"


def test_mapped_entries_have_no_cpu_fallback():
    if S.device_count() > 0:
        pytest.skip("CUDA device present")
    t = R.encode(np.zeros((48000, 2)), S.PCM_S16, 48000)
    with pytest.raises(S.AnalysisError) as e:
        S.loudness_batch_pcm([t], channel_maps=[[F, F]], per_channel=True)
    assert e.value.kind == "ProcessingError" and "no CPU fallback" in e.value.message


# ---- GPU -----------------------------------------------------------------------------------------------------------------
def _full(g: S.Loudness):
    return tuple(v.hex() if isinstance(v, float) else v for v in _fields(g)) + ((g.error.kind, g.error.message) if g.error else (None, None),)


def _all(gs):
    return [(_full(g), [_full(c) for c in g.per_channel] if g.per_channel is not None else None) for g in gs]


def _check(g: S.Loudness, ref: dict, label=""):
    assert g.error is None, f"{label}: {g.error}"
    assert (g.n_momentary, g.n_short_term) == (ref["n_momentary"], ref["n_short_term"]), label
    for f, tol in (("integrated_lufs", 0.01), ("momentary_max_lufs", 0.01), ("short_term_max_lufs", 0.01), ("loudness_range_lu", 0.02)):
        a, b = getattr(g, f), ref[f]
        if math.isinf(b):
            assert a == b, f"{label} {f}: {a} vs {b}"
        else:
            assert abs(a - b) <= tol, f"{label} {f}: {a} vs {b}"
    assert g.sample_peak == ref["sample_peak"], label
    assert abs(g.true_peak - ref["true_peak"]) <= 1e-5 * ref["true_peak"], f"{label} true_peak: {g.true_peak} vs {ref['true_peak']}"


def _batch(sr=48000):
    """1..8 channels over the six formats, with lengths around the block boundaries, a failing track and an empty one."""
    Sb = (sr + 5) // 10
    lengths = [int(0.3 * sr), 4 * Sb, int(2.9 * sr), 30 * Sb + 7, 12 * sr]
    tracks = []
    for i in range(16):
        C_ = 1 + i % 8
        tracks.append(R.encode(_multichannel(C_, lengths[i % len(lengths)], sr, 300 + i), FMTS[i % len(FMTS)], sr))
    tracks.append(S.PcmTrack(tracks[3].data.copy(), tracks[3].fmt, tracks[3].channels, 7999))
    tracks.append(S.PcmTrack(np.zeros(0, np.uint8), S.PCM_S16, 3, sr))
    return tracks


@pytest.mark.gpu
def test_default_class_map_equals_no_map_and_the_existing_entries():
    tracks = _batch()
    ids = [i % 3 if i % 5 else None for i in range(len(tracks))]
    maps = [S.channel_map(0, t.channels) for t in tracks]
    t0, a0 = S.loudness_albums_pcm(tracks, ids)
    t1, a1 = S.loudness_albums_pcm(tracks, ids, channel_maps=maps)
    t2, a2 = S.loudness_albums_pcm(tracks, ids, channel_maps=[None] * len(tracks), per_channel=True)
    assert _all(t1) == _all(t0) and [_full(a) for a in a1] == [_full(a) for a in a0]
    assert [_full(g) for g in t2] == [_full(g) for g in t0] and [_full(a) for a in a2] == [_full(a) for a in a0]
    # the existing C entry, called directly, gives the same bits
    cat = np.concatenate([t.data for t in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    n, na = len(tracks), len(a0)
    res, alb = (S.StratumLoudness * n)(), (S.StratumLoudness * na)()
    idv = np.array([S.NO_ALBUM if a is None else a for a in ids], np.uint32)
    st = S.lib().stratum_b200_loudness_albums_pcm(cat.ctypes.data, offsets.ctypes.data_as(U64P), srs.ctypes.data_as(U32P), chans.ctypes.data_as(U32P),
                                                  fmts.ctypes.data_as(U32P), n, idv.ctypes.data_as(U32P), na, None, 0, res, alb)
    assert st == S.OK
    assert [_full(S._loudness(r)) for r in res] == [_full(g) for g in t0]
    assert [_full(S._loudness(a)) for a in alb] == [_full(a) for a in a0]


LAYOUTS = [("2.1", 0xB, 3, False), ("4.0", 0x107, 4, False), ("5.1-side", 0x60F, 6, False), ("7.1", 0x63F, 8, False), ("dual-mono", 0x4, 1, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [44100, 48000, 96000])
def test_mapped_layouts_match_the_float64_reference(sr):
    tracks, maps = [], []
    for i, (name, mask, C_, dual) in enumerate(LAYOUTS):
        tracks.append(R.encode(_multichannel(C_, int(14.5 * sr), sr, 500 + i), FMTS[(i + 1) % len(FMTS)], sr))
        maps.append(S.channel_map(mask, C_, dual_mono=dual))
    got = S.loudness_batch_pcm(tracks, channel_maps=maps)
    for (name, *_), g, t, m in zip(LAYOUTS, got, tracks, maps):
        _check(g, RL.measure(t, m), f"{name} @ {sr}")


@pytest.mark.gpu
def test_two_one_with_unused_lfe_is_its_stereo_pair():
    sr = 44100
    x = np.concatenate([_stereo_c2(7, 40 * sr, sr), 0.8 * _multichannel(1, 40 * sr, sr, 9)], axis=1)
    t21 = R.encode(x, S.PCM_S24, sr)
    st = R.encode(x[:, :2], S.PCM_S24, sr)
    g21, g0 = S.loudness_batch_pcm([t21, st], channel_maps=[[F, F, U], None])
    for f in ("integrated_lufs", "momentary_max_lufs", "short_term_max_lufs", "loudness_range_lu", "n_momentary", "n_short_term"):
        assert getattr(g21, f) == getattr(g0, f), f
    default = S.loudness_batch_pcm([t21])[0]  # the default map weighs the third channel as a centre
    assert default.integrated_lufs > g21.integrated_lufs
    assert g21.sample_peak >= g0.sample_peak  # the peaks still cover every channel


@pytest.mark.gpu
def test_loud_mono_as_dual_mono_reads_three_db_more():
    sr = 48000
    t = R.encode(0.9 * _multichannel(1, 45 * sr, sr, 17), S.PCM_F32, sr)
    mono, dual = S.loudness_batch_pcm([t, t], channel_maps=[None, S.channel_map(0, 1, dual_mono=True)])
    for f in ("integrated_lufs", "momentary_max_lufs", "short_term_max_lufs"):
        assert abs(getattr(dual, f) - getattr(mono, f) - 10 * math.log10(2)) <= 1e-9, f
    assert abs(dual.loudness_range_lu - mono.loudness_range_lu) <= 1e-9
    assert (dual.sample_peak, dual.true_peak) == (mono.sample_peak, mono.true_peak)


@pytest.mark.gpu
@pytest.mark.parametrize("sr", [44100, 96000])
def test_per_channel_results_are_one_channel_tracks(sr):
    tracks = []
    for i, C_ in enumerate([1, 2, 3, 4, 5, 6, 7, 8, 2, 6, 33]):
        n = int((3.5 + 2.3 * i) * sr) if C_ < 33 else int(4.1 * sr)
        tracks.append(R.encode(_multichannel(C_, n, sr, 700 + i), FMTS[i % len(FMTS)], sr))
    maps = [S.channel_map(m, t.channels) for m, t in zip([0, 0x3, 0xB, 0x33, 0x37, 0x60F, 0x13F, 0x63F, 0, 0x3F, 0], tracks)]
    got = S.loudness_batch_pcm(tracks, channel_maps=maps, per_channel=True)
    plain = S.loudness_batch_pcm(tracks)
    singles = S.loudness_batch_pcm([RL.channel_track(t, c) for t in tracks for c in range(t.channels)])
    at = 0
    for t, g, p in zip(tracks, got, plain):
        assert len(g.per_channel) == t.channels
        assert [_full(c) for c in g.per_channel] == [_full(s) for s in singles[at:at + t.channels]]
        at += t.channels
        assert g.sample_peak == max(c.sample_peak for c in g.per_channel) == p.sample_peak
        assert g.true_peak == max(c.true_peak for c in g.per_channel) == p.true_peak


@pytest.mark.gpu
def test_per_channel_results_of_failed_tracks_carry_the_error():
    sr = 48000
    good = R.encode(_multichannel(2, 3 * sr, sr, 1), S.PCM_S16, sr)
    low = S.PcmTrack(good.data.copy(), S.PCM_S16, 2, 7999)
    empty = S.PcmTrack(np.zeros(0, np.uint8), S.PCM_S16, 3, sr)
    got = S.loudness_batch_pcm([good, low, empty], per_channel=True)
    assert got[0].error is None and all(c.error is None for c in got[0].per_channel)
    for g in got[1:]:
        assert g.error is not None
        assert [(c.error.kind, c.error.message, c.channels, c.sample_rate, c.frames) for c in g.per_channel] == \
            [(g.error.kind, g.error.message, 1, g.sample_rate, g.frames)] * g.channels


@pytest.mark.gpu
def test_mapped_albums_match_the_pooled_reference():
    sr = 48000
    specs = [(44100, 8, 0x63F, 21.0), (48000, 3, 0xB, 12.0), (96000, 1, 0x4, 9.0), (48000, 4, 0x107, 33.0), (44100, 6, 0x60F, 7.0)]
    tracks, maps = [], []
    for i, (r, C_, mask, d) in enumerate(specs):
        tracks.append(R.encode(_multichannel(C_, int(d * r), r, 900 + i), FMTS[i % len(FMTS)], r))
        maps.append(S.channel_map(mask, C_, dual_mono=C_ == 1))
    ids = [0, 1, 0, 1, 0]
    got, albums = S.loudness_albums_pcm(tracks, ids, channel_maps=maps)
    for a in range(2):
        members = [i for i in range(len(tracks)) if ids[i] == a]
        ref = RL.measure_album([tracks[i] for i in members], [maps[i] for i in members])
        _check(albums[a], ref, f"album {a}")
        assert albums[a].frames == ref["frames"]
    _, (one,) = S.loudness_albums_pcm([tracks[0]], [0], channel_maps=[maps[0]])
    keep = [f for f in FIELDS if f not in ("sample_rate", "channels")]
    assert [getattr(one, f) for f in keep] == [getattr(got[0], f) for f in keep]


@pytest.mark.gpu
def test_mapped_results_do_not_depend_on_chunks_entries_or_devices(monkeypatch):
    import torch

    sr = 44100
    tracks = [R.encode(_multichannel(8, 20 * sr, sr, 41), S.PCM_S16, sr), R.encode(_multichannel(1, 9 * 48000, 48000, 42), S.PCM_F32, 48000),
              R.encode(_multichannel(3, 31 * sr, sr, 43), S.PCM_S24, sr), R.encode(_multichannel(6, 5 * 96000, 96000, 44), S.PCM_U8, 96000),
              R.encode(_multichannel(2, 35 * sr, sr, 45), S.PCM_F64, sr)]
    maps = [S.channel_map(0x63F, 8), S.channel_map(0, 1, dual_mono=True), [F, F, U], S.channel_map(0x60F, 6), None]
    ids = [0, 1, 0, None, 1]
    kw = dict(channel_maps=maps, per_channel=True)
    whole_t, whole_a = S.loudness_albums_pcm(tracks, ids, **kw)
    whole = (_all(whole_t), [_full(a) for a in whole_a])
    assert whole_t[0].integrated_lufs != S.loudness_batch_pcm(tracks[:1])[0].integrated_lufs  # the map is in effect
    t, a = S.loudness_albums_pcm(tracks, ids, devices=[0, 0], **kw)
    assert (_all(t), [_full(x) for x in a]) == whole
    monkeypatch.setenv("STRATUM_B200_STAGE_MB", "1")  # every track in an upload chunk of its own
    t, a = S.loudness_albums_pcm(tracks, ids, **kw)
    assert (_all(t), [_full(x) for x in a]) == whole
    res, t, a = S.analyze_loudness_pcm(tracks, albums=ids, **kw)
    assert (_all(t), [_full(x) for x in a]) == whole
    monkeypatch.delenv("STRATUM_B200_STAGE_MB")
    res2, t, a = S.analyze_loudness_pcm(tracks, albums=ids, **kw)
    assert (_all(t), [_full(x) for x in a]) == whole
    ref = S.analyze_batch_pcm(tracks)
    for r in res + res2 + ref:
        r.metadata.processing_time_ms = 0.0
    assert [_py(r) for r in res] == [_py(r) for r in ref] == [_py(r) for r in res2]
    cat = np.concatenate([x.data for x in tracks])
    offsets, srs, chans, fmts = S._pcm_tables(tracks)
    d = torch.from_numpy(cat).cuda()
    t, a = S.loudness_albums_pcm_device(d.data_ptr(), offsets, srs, chans, fmts, ids, device=d.device.index, **kw)
    torch.cuda.synchronize()
    assert (_all(t), [_full(x) for x in a]) == whole
    if S.device_count() >= 2:
        t, a = S.loudness_albums_pcm(tracks, ids, devices=[0, 1], **kw)
        assert (_all(t), [_full(x) for x in a]) == whole


@pytest.mark.gpu
def test_mapped_results_across_two_devices():
    if S.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    sr = 48000
    tracks = [R.encode(_multichannel(2 + 2 * i, (10 + 5 * i) * sr, sr, 60 + i), FMTS[i], sr) for i in range(4)]
    maps = [S.channel_map(0, t.channels) for t in tracks]
    one = S.loudness_batch_pcm(tracks, devices=[0], channel_maps=maps, per_channel=True)
    two = S.loudness_batch_pcm(tracks, devices=[0, 1], channel_maps=maps, per_channel=True)
    assert _all(two) == _all(one)


@pytest.mark.gpu
def test_launches_and_read_backs():
    sr = 48000
    tracks = [R.encode(_multichannel(c, 5 * sr, sr, 31 + c), S.PCM_S16, sr) for c in (2, 6, 8)]
    n, n_ch = len(tracks), sum(t.channels for t in tracks)
    S.loudness_batch_pcm(tracks, per_channel=True)  # buffers sized before counting

    def counted(**kw):
        l0, (_, d0) = S.launch_count(), S.transfer_bytes()
        S.loudness_batch_pcm(tracks, **kw)
        l1, (_, d1) = S.launch_count(), S.transfer_bytes()
        return l1 - l0, d1 - d0

    assert counted() == (4, n * LOUD_OUT_BYTES)  # one chunk: pass 1, scan, pass 2, gate; the track results
    assert counted(channel_maps=[S.channel_map(0x63F if t.channels == 8 else 0, t.channels) for t in tracks]) == (4, n * LOUD_OUT_BYTES)
    assert counted(per_channel=True) == (4, (n + n_ch) * LOUD_OUT_BYTES)  # the channel CTAs ride in the gate launch
