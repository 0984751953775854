#!/usr/bin/env python3
"""Throughput of the loudness measurement (stratum_b200_loudness_batch_pcm) on one GPU.

    python tools/loudness_bench.py [--tracks N] [--rounds R] [--warmup W] [--albums [M]] [--with-analysis] [--devices D] [--out FILE]
    python tools/loudness_bench.py --layout [--tracks N] [--rounds R] [--warmup W] [--out FILE]
    python tools/loudness_bench.py --baseline-lib LIB [--tracks N] [--rounds R] [--warmup W] [--out FILE]
    python tools/loudness_bench.py --series [--tracks N] [--rounds R] [--warmup W] [--out FILE]

Workload: N (default 1024) stereo three-minute 44.1 kHz PCM16 tracks, each channel a C2 track of tests/synth.py (channel 0 from
seed i, channel 1 from seed i + 1000), generated on the device and quantised there.  Two legs (three with --albums), timed in
alternation after W untimed calls of each:
  device  the PCM already in device memory (stratum_b200_loudness_batch_pcm_device);
  host    the same bytes in pinned host memory (stratum_b200_loudness_batch_pcm: upload included);
  albums  with --albums M (default 12): the host leg as albums of M consecutive tracks (stratum_b200_loudness_albums_pcm), which
          adds the read-back of the momentary / short-term powers and the album gate.
With --with-analysis four more legs over the same pinned bytes, run with stage timing off:
  analysis       stratum_b200_analyze_batch_pcm alone (default configuration);
  loudness       stratum_b200_loudness_batch_pcm alone (the host leg without stage timing);
  separate       analysis, then loudness: what a caller wanting both paid before;
  combined       stratum_b200_analyze_loudness_pcm: both from one upload.
Each reports tracks/s, wall time and the host-to-device bytes of one call; one more combined call with stage timing on gives the
loudness kernel times inside it and the analysis stage total beside them.  --devices D runs every host leg over devices 0..D-1 from
this process (the device leg stays on device 0).
--layout measures channel maps instead, on N (default 256) 7.1 three-minute 44.1 kHz PCM16 tracks (about 32 GB; channel c of track i
the C2 track i + 1000 c): three kinds, each device-resident and from pinned host memory, six legs timed in alternation:
  default      no channel map (the default map weighs the 7.1 rear pair as Ls Rs and the side pair 0);
  mapped       the 7.1 map of stratum_b200_loudness_channel_map(0x63F, 8, 0, map) (stratum_b200_loudness_mapped_pcm);
  per_channel  the same map plus per-channel results (the per-channel CTAs of the gate launch and their read-back).
Each leg reports tracks/s, wall time, the median pass 2 and gate kernel times and the device-to-host bytes of one call.
--series measures the loudness series on the default stereo workload: without and with all four series
(stratum_b200_loudness_series_pcm: momentary and short-term loudness, sample and true peaks per 100 ms), each device-resident and
from pinned host memory, four legs timed in alternation; each reports tracks/s, wall time, the median pass 2 and gate kernel times and
the device-to-host bytes of one call.
--baseline-lib LIB times the stereo device leg of this build against another build of the library (e.g. the parent commit's), the
two alternating, and reports each one's median, minimum and maximum pass 2 time and whether the two give the same bits.
Reports the median over R rounds of tracks/s and wall time per leg, the median kernel times of the device leg (pass 1, the scan,
pass 2 with the true-peak FIR, the gate), the album gate's kernel time and the device-to-host bytes the album leg adds to the host
leg (stratum_b200_transfer_bytes), the host-to-device rate of a plain 4 GB pinned copy measured in the same run, and the card's name
and power limit.  Prints one JSON document."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

SR, N_FRAMES = 44100, 7_938_000
STAGES = ("loudness_pass1", "loudness_scan", "loudness_pass2", "loudness_gate")


def card() -> dict:
    import torch

    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                           timeout=10).stdout.strip()
        out["power_limit"], out["sm_max_clock"] = [s.strip() for s in q.split(",")]
    except Exception as e:  # the numbers are still measured; the card line says why it is incomplete
        out["query_error"] = type(e).__name__
    return out


def make_pcm(S, torch, n_tracks: int, C: int = 2):
    """int16 (n_tracks * N_FRAMES * C) on the device: interleaved, channel c of track i = C2 track i + 1000 c."""
    import synth

    pcm = torch.empty(n_tracks * N_FRAMES * C, dtype=torch.int16, device="cuda")
    group = 32 if C <= 2 else 8
    tmp = torch.empty(C * group * N_FRAMES, dtype=torch.float32, device="cuda")
    for g0 in range(0, n_tracks, group):
        n = min(group, n_tracks - g0)
        rows = []
        for c in range(C):
            for i in range(g0, g0 + n):
                p = synth.c2_params(i + 1000 * c, N_FRAMES, SR)
                rows.append([p.bpm, p.tonic, p.minor, p.phase_frac, p.chord_amp])
        S.synth_batch(tmp.data_ptr(), C * n, N_FRAMES, SR, np.asarray(rows, np.float32), 0)
        x = tmp[: C * n * N_FRAMES].view(C, n, N_FRAMES).permute(1, 2, 0)  # (track, frame, channel)
        q = torch.clamp(torch.round(x * 32768.0), -32768, 32767).to(torch.int16)
        pcm[g0 * N_FRAMES * C:(g0 + n) * N_FRAMES * C] = q.reshape(-1)
    del tmp
    torch.cuda.synchronize()
    return pcm


def lib_stage_times(L) -> dict:
    """Stage times of library handle L since its last reset (S.stage_times for another build of the library)."""
    names = C.create_string_buffer(4096)
    ms = (C.c_double * 64)()
    n = L.stratum_b200_stage_times(names, 4096, ms, 64)
    return {nm: ms[i] for i, nm in enumerate([s for s in names.value.decode().split("\n") if s][:n])}


def layout_main(a, S, torch) -> dict:
    n = a.tracks
    L = S.lib()
    d_pcm = make_pcm(S, torch, n, 8)
    h_pcm = torch.empty(d_pcm.numel(), dtype=torch.int16, pin_memory=True)
    h_pcm.copy_(d_pcm)
    bytes_per_track = N_FRAMES * 8 * 2
    offsets = (np.arange(n + 1, dtype=np.uint64) * np.uint64(bytes_per_track))
    srs, chans, fmts = np.full(n, SR, np.uint32), np.full(n, 8, np.uint32), np.full(n, S.PCM_S16, np.uint32)
    u32 = lambda v: v.ctypes.data_as(C.POINTER(C.c_uint32))
    off = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    cmap = np.ascontiguousarray(np.tile(np.asarray(S.channel_map(0x63F, 8), np.uint8), n))
    mp = cmap.ctypes.data_as(C.POINTER(C.c_uint8))
    res = (S.StratumLoudness * n)()
    chout = (S.StratumLoudness * (8 * n))()
    kinds = {"default": (None, None), "mapped": (mp, None), "per_channel": (mp, chout)}

    def leg(kind, where):
        m, co = kinds[kind]
        if where == "device":
            return lambda: L.stratum_b200_loudness_mapped_pcm_device(C.c_void_p(d_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, None, 0, m, 0,
                                                                     res, None, co)
        return lambda: L.stratum_b200_loudness_mapped_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, None, 0, m, None, 0, res,
                                                          None, co)

    legs = {(k, w): leg(k, w) for k in kinds for w in ("device", "host")}

    def timed(fn):
        S.stage_timing(True)
        S.stage_times(reset=True)
        _, d2h0 = S.transfer_bytes()
        t0 = time.perf_counter()
        st = fn()
        wall = time.perf_counter() - t0
        S.stage_timing(False)
        if st != S.OK:
            raise SystemExit(f"loudness call failed: {S.last_error()}")
        _, d2h1 = S.transfer_bytes()
        return wall, S.stage_times(), sum(1 for i in range(n) if res[i].status == 0), d2h1 - d2h0, res[0].integrated_lufs

    for _ in range(a.warmup):
        for fn in legs.values():
            timed(fn)
    runs = {key: [] for key in legs}
    for _ in range(a.rounds):
        for key, fn in legs.items():
            runs[key].append(timed(fn))
    doc = {"workload": f"{n} 7.1 (8-channel) 3-minute 44.1 kHz PCM16 tracks (synthetic C2 tracks per channel)", "card": card(), "rounds": a.rounds,
           "warmup": a.warmup, "pcm_bytes": n * bytes_per_track, "map": S.channel_map(0x63F, 8)}
    for (kind, where), rs in runs.items():
        wall = statistics.median(r[0] for r in rs)
        doc[f"{kind}_{where}"] = {"tracks_per_s": n / wall, "wall_s": wall,
                                  "stage_ms": {s: statistics.median(r[1].get(s, 0.0) for r in rs) for s in STAGES},
                                  "d2h_bytes": statistics.median(r[3] for r in rs), "ok_tracks": min(r[2] for r in rs), "track0_integrated_lufs": rs[-1][4]}
    return doc


def series_main(a, S, torch) -> dict:
    n = a.tracks
    L = S.lib()
    d_pcm = make_pcm(S, torch, n)
    h_pcm = torch.empty(d_pcm.numel(), dtype=torch.int16, pin_memory=True)
    h_pcm.copy_(d_pcm)
    bytes_per_track = N_FRAMES * 2 * 2
    offsets = (np.arange(n + 1, dtype=np.uint64) * np.uint64(bytes_per_track))
    srs, chans, fmts = np.full(n, SR, np.uint32), np.full(n, 2, np.uint32), np.full(n, S.PCM_S16, np.uint32)
    u32 = lambda v: v.ctypes.data_as(C.POINTER(C.c_uint32))
    off = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    _, arrays = S._series_args(True, offsets, srs, chans, fmts)
    ptrs = [x.ctypes.data_as(C.POINTER(C.c_double)) for x in arrays]
    res = (S.StratumLoudness * n)()
    kinds = {"plain": [None] * 4, "series": ptrs}

    def leg(kind, where):
        p = kinds[kind]
        if where == "device":
            return lambda: L.stratum_b200_loudness_series_pcm_device(C.c_void_p(d_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, None, 0, None, 0,
                                                                     res, None, None, *p)
        return lambda: L.stratum_b200_loudness_series_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, None, 0, None, None, 0, res,
                                                          None, None, *p)

    legs = {(k, w): leg(k, w) for k in kinds for w in ("device", "host")}

    def timed(fn):
        S.stage_timing(True)
        S.stage_times(reset=True)
        _, d2h0 = S.transfer_bytes()
        t0 = time.perf_counter()
        st = fn()
        wall = time.perf_counter() - t0
        S.stage_timing(False)
        if st != S.OK:
            raise SystemExit(f"loudness call failed: {S.last_error()}")
        _, d2h1 = S.transfer_bytes()
        return wall, S.stage_times(), sum(1 for i in range(n) if res[i].status == 0), d2h1 - d2h0

    for _ in range(a.warmup):
        for fn in legs.values():
            timed(fn)
    runs = {key: [] for key in legs}
    for _ in range(a.rounds):
        for key, fn in legs.items():
            runs[key].append(timed(fn))
    doc = {"workload": f"{n} stereo 3-minute 44.1 kHz PCM16 tracks (synthetic C2 pairs)", "card": card(), "rounds": a.rounds, "warmup": a.warmup,
           "pcm_bytes": n * bytes_per_track, "series_entries": {k: int(x.size) for k, x in zip(("momentary", "short_term", "sample_peak", "true_peak"), arrays)},
           "track0": {"momentary_max_lufs": res[0].momentary_max_lufs, "series_momentary_max_lufs": float(arrays[0][:res[0].n_momentary].max()),
                      "true_peak": res[0].true_peak, "series_true_peak": float(arrays[3][:len(arrays[3]) // n].max())}}
    for (kind, where), rs in runs.items():
        wall = statistics.median(r[0] for r in rs)
        doc[f"{kind}_{where}"] = {"tracks_per_s": n / wall, "wall_s": wall,
                                  "stage_ms": {s: statistics.median(r[1].get(s, 0.0) for r in rs) for s in STAGES},
                                  "d2h_bytes": statistics.median(r[3] for r in rs), "ok_tracks": min(r[2] for r in rs)}
    return doc


def baseline_main(a, S, torch) -> dict:
    """The stereo device leg of this build and of the library at a.baseline_lib, alternating."""
    n = a.tracks
    L = S.lib()
    B = C.CDLL(str(Path(a.baseline_lib).resolve()))
    B.stratum_b200_loudness_batch_pcm_device.argtypes = L.stratum_b200_loudness_batch_pcm_device.argtypes
    B.stratum_b200_loudness_batch_pcm_device.restype = C.c_int32
    B.stratum_b200_stage_times.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_double), C.c_int32]
    B.stratum_b200_stage_times.restype = C.c_int32
    B.stratum_b200_stage_timing_enable.argtypes = [C.c_int32]
    d_pcm = make_pcm(S, torch, n)
    offsets = (np.arange(n + 1, dtype=np.uint64) * np.uint64(N_FRAMES * 2 * 2))
    srs, chans, fmts = np.full(n, SR, np.uint32), np.full(n, 2, np.uint32), np.full(n, S.PCM_S16, np.uint32)
    u32 = lambda v: v.ctypes.data_as(C.POINTER(C.c_uint32))
    off = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    out = {"this": (S.StratumLoudness * n)(), "baseline": (S.StratumLoudness * n)()}
    libs = {"this": L, "baseline": B}

    def timed(key):
        lb = libs[key]
        lb.stratum_b200_stage_timing_enable(1)
        lb.stratum_b200_stage_times_reset()
        t0 = time.perf_counter()
        st = lb.stratum_b200_loudness_batch_pcm_device(C.c_void_p(d_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, 0, out[key])
        wall = time.perf_counter() - t0
        lb.stratum_b200_stage_timing_enable(0)
        if st != S.OK:
            raise SystemExit(f"{key}: loudness call failed")
        return wall, lib_stage_times(lb)

    for _ in range(a.warmup):
        for key in libs:
            timed(key)
    runs = {key: [] for key in libs}
    for _ in range(a.rounds):
        for key in libs:
            runs[key].append(timed(key))
    same = C.string_at(C.addressof(out["this"]), C.sizeof(out["this"])) == C.string_at(C.addressof(out["baseline"]), C.sizeof(out["baseline"]))
    doc = {"workload": f"{n} stereo 3-minute 44.1 kHz PCM16 tracks (synthetic C2 pairs), device-resident", "card": card(), "rounds": a.rounds,
           "warmup": a.warmup, "baseline_lib": Path(a.baseline_lib).name, "results_bit_identical": same}
    for key, rs in runs.items():
        p2 = [r[1].get("loudness_pass2", 0.0) for r in rs]
        doc[key] = {"wall_s": statistics.median(r[0] for r in rs), "pass2_ms": {"median": statistics.median(p2), "min": min(p2), "max": max(p2)},
                    "stage_ms": {s: statistics.median(r[1].get(s, 0.0) for r in rs) for s in STAGES}}
    return doc


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=None, help="default 1024 (256 with --layout)")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--albums", type=int, nargs="?", const=12, default=None, metavar="M", help="add the album leg, M tracks per album")
    ap.add_argument("--with-analysis", action="store_true", help="add the analysis, separate and combined legs")
    ap.add_argument("--devices", type=int, default=1, help="host legs over devices 0..D-1")
    ap.add_argument("--layout", action="store_true", help="time channel maps and per-channel results on 7.1 tracks")
    ap.add_argument("--series", action="store_true", help="time the loudness series against the plain measurement")
    ap.add_argument("--baseline-lib", default=None, metavar="LIB", help="time the stereo device leg of this build against the library LIB")
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    a = ap.parse_args()
    a.tracks = a.tracks or (256 if a.layout else 1024)
    import torch

    import stratum_dsp_b200 as S

    if not torch.cuda.is_available() or S.device_count() < 1:
        raise SystemExit("loudness_bench needs a CUDA device: the measurement has no CPU fallback")
    if a.layout or a.baseline_lib or a.series:
        doc = layout_main(a, S, torch) if a.layout else (series_main(a, S, torch) if a.series else baseline_main(a, S, torch))
        s = json.dumps(doc, indent=1)
        print(s)
        if a.out:
            Path(a.out).parent.mkdir(parents=True, exist_ok=True)
            Path(a.out).write_text(s + "\n")
        return
    if not 1 <= a.devices <= S.device_count():
        raise SystemExit(f"--devices {a.devices}: {S.device_count()} CUDA device(s) present")
    n = a.tracks
    L = S.lib()
    d_pcm = make_pcm(S, torch, n)
    h_pcm = torch.empty(d_pcm.numel(), dtype=torch.int16, pin_memory=True)
    h_pcm.copy_(d_pcm)
    bytes_per_track = N_FRAMES * 2 * 2
    offsets = (np.arange(n + 1, dtype=np.uint64) * np.uint64(bytes_per_track))
    srs = np.full(n, SR, np.uint32)
    chans = np.full(n, 2, np.uint32)
    fmts = np.full(n, S.PCM_S16, np.uint32)
    res = (S.StratumLoudness * n)()
    u32 = lambda v: v.ctypes.data_as(C.POINTER(C.c_uint32))
    off = offsets.ctypes.data_as(C.POINTER(C.c_uint64))
    devs = (C.c_int32 * a.devices)(*range(a.devices))
    nd = a.devices if a.devices > 1 else 0
    devp = devs if nd else None

    def device_leg():
        return L.stratum_b200_loudness_batch_pcm_device(C.c_void_p(d_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, 0, res)

    def host_leg():
        return L.stratum_b200_loudness_batch_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, devp, nd, res)

    n_albums = (n + a.albums - 1) // a.albums if a.albums else 0
    album_of = np.arange(n, dtype=np.uint32) // np.uint32(a.albums or 1)
    alb = (S.StratumLoudness * max(n_albums, 1))()

    def album_leg():
        return L.stratum_b200_loudness_albums_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, u32(album_of), n_albums, devp, nd,
                                                  res, alb)

    ares = (S.StratumResult * n)()
    a_ok = [0]

    def analysis_leg():  # results are counted and released inside the call's wall time: analyze_batch_pcm does the same
        st = L.stratum_b200_analyze_batch_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), C.c_uint32(n), None, devp, C.c_uint32(nd),
                                              ares)
        a_ok[0] = sum(1 for i in range(n) if ares[i].status == 0)
        L.stratum_b200_result_free(ares, n)
        return st

    def separate_leg():
        st = analysis_leg()
        return st if st != S.OK else host_leg()

    def combined_leg():
        st = L.stratum_b200_analyze_loudness_pcm(C.c_void_p(h_pcm.data_ptr()), off, u32(srs), u32(chans), u32(fmts), n, None, None, 0, devp, nd, ares, res, None)
        a_ok[0] = sum(1 for i in range(n) if ares[i].status == 0)
        L.stratum_b200_result_free(ares, n)
        return st

    analysis_legs = (analysis_leg, separate_leg, combined_leg) if a.with_analysis else ()

    def timed(fn, stage_timing=True):
        S.stage_timing(stage_timing)
        S.stage_times(reset=True)
        h2d0, d2h0 = S.transfer_bytes()
        t0 = time.perf_counter()
        st = fn()
        wall = time.perf_counter() - t0
        S.stage_timing(False)
        if st != S.OK:
            raise SystemExit(f"loudness call failed: {S.last_error()}")
        ok = sum(1 for i in range(n) if res[i].status == 0)
        h2d1, d2h1 = S.transfer_bytes()
        return wall, S.stage_times(), ok, d2h1 - d2h0, h2d1 - h2d0, a_ok[0]

    legs = [device_leg, host_leg] + ([album_leg] if n_albums else [])
    for _ in range(a.warmup):
        for fn in legs + list(analysis_legs):
            timed(fn, False)
    runs = {fn: [] for fn in legs}
    plain = {fn: [] for fn in (analysis_leg, "loudness", separate_leg, combined_leg)} if analysis_legs else {}
    for _ in range(a.rounds):
        for fn in legs:
            runs[fn].append(timed(fn))
        if analysis_legs:  # alternated: analysis, loudness, separate, combined
            plain[analysis_leg].append(timed(analysis_leg, False))
            plain["loudness"].append(timed(host_leg, False))
            plain[separate_leg].append(timed(separate_leg, False))
            plain[combined_leg].append(timed(combined_leg, False))
    profile = timed(combined_leg) if analysis_legs else None
    dev, host = runs[device_leg], runs[host_leg]
    # plain pinned host-to-device copy of 4 GB in the same run
    probe = min(h_pcm.numel(), 2 << 30)
    dst = torch.empty(probe, dtype=torch.int16, device="cuda")
    rates = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dst.copy_(h_pcm[:probe], non_blocking=True)
        torch.cuda.synchronize()
        rates.append(probe * 2 / (time.perf_counter() - t0) / 1e9)
    sample = res[0]
    doc = {
        "workload": f"{n} stereo 3-minute 44.1 kHz PCM16 tracks (synthetic C2 pairs)",
        "card": card(),
        "rounds": a.rounds,
        "warmup": a.warmup,
        "device": {"tracks_per_s": n / statistics.median(r[0] for r in dev), "wall_s": statistics.median(r[0] for r in dev),
                   "stage_ms": {s: statistics.median(r[1].get(s, 0.0) for r in dev) for s in STAGES}, "ok_tracks": min(r[2] for r in dev)},
        "host_pinned": {"tracks_per_s": n / statistics.median(r[0] for r in host), "wall_s": statistics.median(r[0] for r in host),
                        "pcm_gb_per_s": n * bytes_per_track / statistics.median(r[0] for r in host) / 1e9, "ok_tracks": min(r[2] for r in host)},
        "h2d_pinned_copy_gb_per_s": statistics.median(rates),
        "track0": {"integrated_lufs": sample.integrated_lufs, "loudness_range_lu": sample.loudness_range_lu, "true_peak": sample.true_peak},
    }
    if n_albums:
        al = runs[album_leg]
        doc["host_albums"] = {"tracks_per_album": a.albums, "albums": n_albums, "tracks_per_s": n / statistics.median(r[0] for r in al),
                              "wall_s": statistics.median(r[0] for r in al), "album_gate_ms": statistics.median(r[1].get("loudness_album_gate", 0.0) for r in al),
                              "extra_d2h_bytes": statistics.median(r[3] for r in al) - statistics.median(r[3] for r in host),
                              "pcm_bytes": n * bytes_per_track, "ok_tracks": min(r[2] for r in al),
                              "ok_albums": sum(1 for i in range(n_albums) if alb[i].status == 0),
                              "album0": {"integrated_lufs": alb[0].integrated_lufs, "loudness_range_lu": alb[0].loudness_range_lu}}
    if a.devices > 1:
        doc["host_devices"] = a.devices
    if analysis_legs:
        def leg(rs):
            wall = statistics.median(r[0] for r in rs)
            return {"tracks_per_s": n / wall, "wall_s": wall, "h2d_bytes": statistics.median(r[4] for r in rs)}

        an = {"analysis": leg(plain[analysis_leg]), "loudness": leg(plain["loudness"]), "separate": leg(plain[separate_leg]),
              "combined": leg(plain[combined_leg])}
        an["analysis"]["ok_tracks"] = min(r[5] for r in plain[analysis_leg])
        an["combined"]["ok_tracks"] = min(r[5] for r in plain[combined_leg])
        an["combined"]["ok_loudness_tracks"] = min(r[2] for r in plain[combined_leg])
        st = profile[1]
        an["combined_profile"] = {"loudness_stage_ms": {s: st.get(s, 0.0) for s in STAGES},
                                  "analysis_stage_ms_sum": sum(v for k, v in st.items() if not k.startswith(("loudness", "host_"))),
                                  "wall_s": profile[0]}
        an["pcm_bytes"] = n * bytes_per_track
        an["combined_vs_separate"] = an["separate"]["wall_s"] / an["combined"]["wall_s"]
        an["combined_vs_analysis"] = an["analysis"]["wall_s"] / an["combined"]["wall_s"]
        doc["with_analysis"] = an
    s = json.dumps(doc, indent=1)
    print(s)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(s + "\n")


if __name__ == "__main__":
    main()
