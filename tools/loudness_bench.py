#!/usr/bin/env python3
"""Throughput of the loudness measurement (stratum_b200_loudness_batch_pcm) on one GPU.

    python tools/loudness_bench.py [--tracks N] [--rounds R] [--warmup W] [--albums [M]] [--with-analysis] [--devices D] [--out FILE]

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


def make_pcm(S, torch, n_tracks: int):
    """int16 (n_tracks * N_FRAMES * 2) on the device: interleaved stereo, channel c of track i = C2 track i + 1000 c."""
    import synth

    pcm = torch.empty(n_tracks * N_FRAMES * 2, dtype=torch.int16, device="cuda")
    group = 32
    tmp = torch.empty(2 * group * N_FRAMES, dtype=torch.float32, device="cuda")
    for g0 in range(0, n_tracks, group):
        n = min(group, n_tracks - g0)
        rows = []
        for c in range(2):
            for i in range(g0, g0 + n):
                p = synth.c2_params(i + 1000 * c, N_FRAMES, SR)
                rows.append([p.bpm, p.tonic, p.minor, p.phase_frac, p.chord_amp])
        S.synth_batch(tmp.data_ptr(), 2 * n, N_FRAMES, SR, np.asarray(rows, np.float32), 0)
        x = tmp[: 2 * n * N_FRAMES].view(2, n, N_FRAMES).permute(1, 2, 0)  # (track, frame, channel)
        q = torch.clamp(torch.round(x * 32768.0), -32768, 32767).to(torch.int16)
        pcm[g0 * N_FRAMES * 2:(g0 + n) * N_FRAMES * 2] = q.reshape(-1)
    del tmp
    torch.cuda.synchronize()
    return pcm


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--tracks", type=int, default=1024)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--albums", type=int, nargs="?", const=12, default=None, metavar="M", help="add the album leg, M tracks per album")
    ap.add_argument("--with-analysis", action="store_true", help="add the analysis, separate and combined legs")
    ap.add_argument("--devices", type=int, default=1, help="host legs over devices 0..D-1")
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    a = ap.parse_args()
    import torch

    import stratum_dsp_b200 as S

    if not torch.cuda.is_available() or S.device_count() < 1:
        raise SystemExit("loudness_bench needs a CUDA device: the measurement has no CPU fallback")
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
