#!/usr/bin/env python3
"""Cost of fine BPM grids on one GPU: tracks/s of the device-resident batch at several min_bpm / max_bpm / bpm_resolution settings.

    python tools/bpm_grid_bench.py [--table bpm|frame] [--rounds R] [--warmup W] [--tracks N] [--out FILE]

Workloads are bench.py's (imported, not copied): C2 = 1024 synthetic three-minute 44.1 kHz tracks generated on the device, timed
at the default grid (40..240 step 1, 201 hypotheses), 40..300 step 1 (261), step 0.1 (2000) and step 0.01 (20006); C4 = one
60-minute mix at the default grid and at 0.01.  The grids of a workload are timed in alternation (one call of each per round,
after W untimed calls of each), so drift of the shared machine spreads over all of them.  Per grid it reports the median
tracks/s over the rounds, the median device time of the call, and the median stage times of the autocorrelation-tempogram
stages ("tempogram": base slot; "multires_tempogram": the escalated hop-256 / hop-1024 slots) and of the legacy estimator
("legacy_bpm", comb filterbank included), with the card's name and power limit read in the same run.  Prints one JSON document.

--table frame times frame_size 2048 (default), 4096 and 8192 on the same workloads instead, with the stage times of the tempo-path
STFT and its feature kernels ("stft_2048_hop512" and "spec_features": base slot; "stft_multires" and "multires_features": the
escalated slots; the stage names keep "2048" at every frame size)."""
from __future__ import annotations

import argparse
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

import bench  # noqa: E402  (workload_layout, fill_device)

GRIDS = {
    "c2": [("40-240/1 (default)", {}), ("40-300/1", {"max_bpm": 300.0}), ("40-240/0.1", {"bpm_resolution": 0.1}),
           ("40-240/0.01", {"bpm_resolution": 0.01})],
    "c4": [("40-240/1 (default)", {}), ("40-240/0.01", {"bpm_resolution": 0.01})],
}
STAGES = ("tempogram", "multires_tempogram", "legacy_bpm")
FRAMES = {wl: [("2048 (default)", {}), ("4096", {"frame_size": 4096}), ("8192", {"frame_size": 8192})] for wl in ("c2", "c4")}
FRAME_STAGES = ("stft_2048_hop512", "spec_features", "stft_multires", "multires_features")
TABLES = {"bpm": (GRIDS, STAGES), "frame": (FRAMES, FRAME_STAGES)}


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


def run_workload(S, torch, wl: str, n_tracks: int, rounds: int, warmup: int, table: str = "bpm") -> dict:
    settings, stages = TABLES[table]
    lens, srs, rows, _ = bench.workload_layout(wl, 0, n_tracks)
    offsets = np.zeros(n_tracks + 1, np.uint64)
    offsets[1:] = np.cumsum(lens, dtype=np.uint64)
    buf = torch.empty(int(offsets[-1]), dtype=torch.float32, device="cuda")
    bench.fill_device(S, torch, wl, buf, offsets, lens, srs, rows, 0)
    grids = [(name, S.AnalysisConfig(**kw) if kw else None) for name, kw in settings[wl]]

    def call(cfg):
        S.stage_times(reset=True)
        t0 = time.perf_counter()
        res = S.analyze_batch_device(buf.data_ptr(), offsets, srs, cfg, 0, convert=False)
        wall = time.perf_counter() - t0
        dev_ms = S.last_call_device_ms()
        ok = sum(1 for r in res if r.status == 0)
        S.free_results(res)
        return wall, dev_ms, S.stage_times(), ok

    for _ in range(warmup):
        for _, cfg in grids:
            call(cfg)
    S.stage_timing(True)
    samples = {name: [] for name, _ in grids}
    for _ in range(rounds):
        for name, cfg in grids:
            samples[name].append(call(cfg))
    S.stage_timing(False)
    del buf
    torch.cuda.empty_cache()
    out = {}
    for name, _ in grids:
        rs = samples[name]
        wall = statistics.median(r[0] for r in rs)
        out[name] = {
            "tracks_per_s": n_tracks / wall,
            "wall_s": wall,
            "device_ms": statistics.median(r[1] for r in rs),
            "stage_ms": {st: statistics.median(r[2].get(st, 0.0) for r in rs) for st in stages},
            "ok_tracks": min(r[3] for r in rs),
        }
    return {"tracks": n_tracks, "rounds": rounds, "warmup": warmup, "grids": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--table", choices=sorted(TABLES), default="bpm", help="bpm: BPM grids; frame: frame_size 2048 / 4096 / 8192")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--tracks", type=int, default=1024, help="C2 batch size")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--out", default=None, help="also write the JSON document to this file")
    args = ap.parse_args()
    import torch
    import stratum_dsp_b200 as S

    if not torch.cuda.is_available():
        raise SystemExit("bpm_grid_bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(0)
    doc = {"card": card(), "table": args.table, "c2": run_workload(S, torch, "c2", args.tracks, args.rounds, args.warmup, args.table)}
    if not args.no_c4:
        doc["c4"] = run_workload(S, torch, "c4", 1, args.rounds, args.warmup, args.table)
    txt = json.dumps(doc, indent=1)
    print(txt)
    if args.out:
        Path(args.out).write_text(txt + "\n")


if __name__ == "__main__":
    main()
